// select_kernels.cuh -- everything around the scoring kernel: corpus/query preparation
// (bf16 shadow + rigorous error bound), the per-slab threshold refresh (radix select over a
// query's candidate list), the fp32 rescore + final sort, the exact fp32 path used as the
// overflow fallback, and the multi-shard merge.
//
// Together with coarse_kernel.cuh these replace faiss's result handlers
// (HeapBlockResultHandler / ReservoirBlockResultHandler, SURVEY.md 3.2) that the reference
// reaches through src/index.py:42.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <float.h>
#include "keys.cuh"
#include "ptx_sm100.cuh"

namespace b2ip {

constexpr int SEL_THREADS = 256;
constexpr int SORT_CAP = 4096;       // u64 keys sorted in shared memory by finalize
constexpr int REFRESH_SMEM_KEYS = 4096;   // candidate lists up to this size are refreshed from smem
constexpr int BOOT_MAX_GROUPS = 160 * 128;   // group maxima per query of the threshold bootstrap (80 KB of smem)
static_assert(REFRESH_SMEM_KEYS <= SORT_CAP, "finalize stages the fused refresh in its sort buffer");
constexpr int FLAG_OVERFLOW = 1;
constexpr int EXACT_QB = 8;          // queries per pass of the exact path
constexpr int RESCORE_JU = 8;        // finalize: float4 chunks per lane held in registers per row (d <= 1024)

// device-side counters of one search (int64 each)
enum { GS_MAX_KEPT = 0, GS_OVERFLOW = 1, GS_CANDIDATES = 2, GS_RESCORED = 3, GS_XSTATUS = 4,
       GS_MAX_ERR = 5,      // run-time certificate: max over rescored rows of |coarse - exact| / eps_q (float bits)
       GS_VIOLATIONS = 6,   // rescored rows with |coarse - exact| > eps_q (must stay 0)
       GS_COUNT = 7 };
constexpr int MAX_PEERS = 8;         // ranks of one NVSwitch box in the peer-direct exchange
constexpr long long XSTATUS_TIMEOUT = 1ll << 40;   // GS_XSTATUS: a peer's flag never arrived
// Flag array of one parity: XF_WORDS uint32 per rank.  Rank r publishes into words
// [XF_WORDS*r ...) of EVERY rank's array.
constexpr int XF_WORDS = 4;
enum { XF_RESULT = 0,     // = seq once rank r's result blocks of search `seq` are in my gather buffer
       XF_OVERFLOW = 1,   // rank r's overflowed queries in that search
       XF_THR = 2 };      // = seq once rank r's per-query bounds are in my threshold buffer

__device__ __forceinline__ unsigned long long global_timer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// Threads 0..world-1 of the block wait until word `word` of every rank's flag group has reached
// `seq` (acquire, system scope), bounded by `timeout_ns` of wall time: a dead peer must not hang
// the GPU -- it leaves XSTATUS_TIMEOUT in *xstatus and the call fails on the host.  Ends with a
// block barrier.
__device__ __forceinline__ void wait_peer_flags(const unsigned int* flags, int world, int word,
                                                unsigned int seq, long long timeout_ns,
                                                long long* xstatus) {
    if (threadIdx.x < world) {
        const unsigned int* f = flags + XF_WORDS * threadIdx.x + word;
        unsigned int v;
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
        if (static_cast<int>(v - seq) < 0) {
            const unsigned long long t0 = global_timer_ns();
            for (;;) {
                __nanosleep(200);
                asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
                if (static_cast<int>(v - seq) >= 0) break;
                if (static_cast<long long>(global_timer_ns() - t0) > timeout_ns) {
                    if (xstatus) atomicMax(xstatus, XSTATUS_TIMEOUT);
                    break;
                }
            }
        }
    }
    __syncthreads();
}

// Per-call values of a search whose launch sequence is replayed from a CUDA graph (small query
// batches): the graph's kernel nodes keep their baked parameters and read what changes from one
// call to the next -- caller buffers, exchange sequence number -- from this device-resident block,
// which the host refreshes with one small copy ahead of the graph launch.  nullptr = use the
// kernel's own parameters.
struct DynArgs {
    const float* q32;        // caller's fp32 queries
    float* out_s;            // caller's result buffers (plain search)
    long long* out_r;
    float* ex_out_s;         // merged results of the peer-direct exchange
    long long* ex_out_r;
    unsigned int seq;        // exchange sequence number
    unsigned int pad;
};

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---------------------------------------------------------------------------------------
// 16-bit operand formats of the coarse GEMM ("shadow" rows / queries)
// ---------------------------------------------------------------------------------------
// SH_BF16: 8 exponent bits, never overflows for fp32 inputs below 3.39e38.
// SH_F16 : 3 more mantissa bits (an 8x tighter error bound on normalised embeddings, and
//          LOSSLESS for the reference's default fp16 embedding shards); values are saturated to
//          +-65504 so the shadow never holds an infinity the input did not have -- the error
//          bound is computed from the value actually stored, so saturation only loosens it.
enum { SH_BF16 = 0, SH_F16 = 1 };

__device__ __forceinline__ float sat_f16(float v) {
    // finite values saturate; NaN and +-inf pass through unchanged (a row that scores inf in
    // fp32 must score inf in the coarse pass too)
    return (fabsf(v) <= FLT_MAX) ? fminf(fmaxf(v, -65504.f), 65504.f) : v;
}
__device__ __forceinline__ bool finite4(float4 v) {
    return fabsf(v.x) <= FLT_MAX && fabsf(v.y) <= FLT_MAX && fabsf(v.z) <= FLT_MAX && fabsf(v.w) <= FLT_MAX;
}
__device__ __forceinline__ uint32_t pack2_sh(float a, float b, int sh) {
    if (sh == SH_F16) {
        const __half2 h = __floats2half2_rn(sat_f16(a), sat_f16(b));
        return *reinterpret_cast<const uint32_t*>(&h);
    }
    const __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<const uint32_t*>(&v);
}
__device__ __forceinline__ float2 unpack2_sh(uint32_t raw, int sh) {
    if (sh == SH_F16) return __half22float2(*reinterpret_cast<const __half2*>(&raw));
    return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&raw));
}
// the same with the element type known at compile time; bf16 -> fp32 is a shift / a mask per element
template <int kSh>
__device__ __forceinline__ float2 unpack2_t(uint32_t raw) {
    if constexpr (kSh == SH_F16) return __half22float2(*reinterpret_cast<const __half2*>(&raw));
    else return make_float2(__uint_as_float(raw << 16), __uint_as_float(raw & 0xFFFF0000u));
}

// ---------------------------------------------------------------------------------------
// corpus ingest
// ---------------------------------------------------------------------------------------
__global__ void widen_f16_kernel(const __half* __restrict__ src, float* __restrict__ dst,
                                 long long count) {
    long long i = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) * 2;
    const long long step = static_cast<long long>(gridDim.x) * blockDim.x * 2;
    for (; i + 1 < count; i += step) {
        const float2 f = __half22float2(*reinterpret_cast<const __half2*>(src + i));
        *reinterpret_cast<float2*>(dst + i) = f;
    }
    if (i < count && i + 1 >= count) dst[i] = __half2float(src[i]);
}

// One warp per row: 16-bit shadow (zero padded to d_pad) + max ||x||^2 and max ||x - sh(x)||^2
// over all rows, which feed the per-query error bound of the coarse scores.
// `src` points at the fp32 rows of [row0,row1) (src_row0 = index of its first row): the master
// rows themselves (fp32 storage) or a staging chunk (16-bit storage, count_delta = false: the
// stored value IS the rounded one, so x - sh(x) is zero by definition).
__global__ void shadow_rows_kernel(const float* __restrict__ src, long long src_row0,
                                   __nv_bfloat16* __restrict__ x16,
                                   long long row0, long long row1, int d, int d_pad,
                                   unsigned int* __restrict__ norm_stats, bool count_delta, int sh) {
    const int lane = threadIdx.x & 31;
    const long long warp = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
    float mx = 0.f, md = 0.f;
    for (long long r = row0 + warp; r < row1; r += nwarps) {
        const float4* srow = reinterpret_cast<const float4*>(src + (r - src_row0) * d);
        uint2* dst = reinterpret_cast<uint2*>(x16 + r * d_pad);
        float nx = 0.f, nd = 0.f;
        bool ok = true;
        for (int j = lane; j < d_pad / 4; j += 32) {
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (j < d / 4) v = __ldg(srow + j);
            ok = ok && finite4(v);
            uint2 o;
            o.x = pack2_sh(v.x, v.y, sh);
            o.y = pack2_sh(v.z, v.w, sh);
            const float2 flo = unpack2_sh(o.x, sh), fhi = unpack2_sh(o.y, sh);
            const float e0 = v.x - flo.x, e1 = v.y - flo.y, e2 = v.z - fhi.x, e3 = v.w - fhi.y;
            if (!count_delta) v = make_float4(flo.x, flo.y, fhi.x, fhi.y);
            nx += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
            nd += e0 * e0 + e1 * e1 + e2 * e2 + e3 * e3;
            dst[j] = o;
        }
        nx = warp_sum(nx);
        nd = warp_sum(nd);
        // Rows with a NaN / inf ELEMENT stay out of the bound: their coarse score is NaN / +-inf
        // exactly when their fp32 score is, so they need no error margin (NaN never reports,
        // +inf always does and is rescored).  A finite row whose norm overflows stays in: the
        // bound becomes inf and the affected queries take the exact path.
        if (__all_sync(0xffffffffu, ok)) {
            mx = fmaxf(mx, nx);
            if (count_delta) md = fmaxf(md, nd);
        }
    }
    if (lane == 0) {
        // non-negative floats order like their bit patterns
        atomicMax(norm_stats + 0, __float_as_uint(mx));
        atomicMax(norm_stats + 1, __float_as_uint(md));
    }
}

// 16-bit rows handed in in the storage type itself (bf16 -> bf16 store, fp16 -> fp16 store):
// copy into the padded layout + max ||x||^2.  One warp per row.
__global__ void ingest_16bit_rows_kernel(const __nv_bfloat16* __restrict__ src,
                                         __nv_bfloat16* __restrict__ x16, long long row0,
                                         long long row1, int d, int d_pad,
                                         unsigned int* __restrict__ norm_stats, int sh) {
    const int lane = threadIdx.x & 31;
    const long long warp = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
    float mx = 0.f;
    for (long long r = row0 + warp; r < row1; r += nwarps) {
        const uint32_t* srow = reinterpret_cast<const uint32_t*>(src + (r - row0) * d);
        uint32_t* dst = reinterpret_cast<uint32_t*>(x16 + r * d_pad);
        float nx = 0.f;
        bool ok = true;
        for (int j = lane; j < d_pad / 2; j += 32) {
            uint32_t v = 0u;
            if (j < d / 2) v = srow[j];
            const float2 f = unpack2_sh(v, sh);
            ok = ok && fabsf(f.x) <= FLT_MAX && fabsf(f.y) <= FLT_MAX;
            nx += f.x * f.x + f.y * f.y;
            dst[j] = v;
        }
        nx = warp_sum(nx);
        if (__all_sync(0xffffffffu, ok)) mx = fmaxf(mx, nx);
    }
    if (lane == 0) atomicMax(norm_stats + 0, __float_as_uint(mx));
}

__global__ void widen_16bit_rows_kernel(const __nv_bfloat16* __restrict__ x16, long long row0,
                                        long long n, int d, int d_pad, float* __restrict__ out,
                                        int sh) {
    const long long total = n * d;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const long long r = i / d;
        const int j = static_cast<int>(i - r * d);
        const unsigned short raw = reinterpret_cast<const unsigned short*>(x16)[(row0 + r) * d_pad + j];
        out[i] = unpack2_sh(raw, sh).x;
    }
}

// One corpus row as 4 consecutive floats starting at element 4*j4, from either storage.
__device__ __forceinline__ float4 load_row4(const float* __restrict__ x32,
                                            const __nv_bfloat16* __restrict__ x16, long long row,
                                            int d, int d_pad, int j4, int sh) {
    if (x32) return __ldg(reinterpret_cast<const float4*>(x32 + row * d) + j4);
    const uint2 raw = __ldg(reinterpret_cast<const uint2*>(x16 + row * d_pad) + j4);
    const float2 lo = unpack2_sh(raw.x, sh), hi = unpack2_sh(raw.y, sh);
    return make_float4(lo.x, lo.y, hi.x, hi.y);
}

// ---------------------------------------------------------------------------------------
// query preparation: 16-bit copy + eps2[q] = 2 * bound(|coarse - exact|), state reset
// ---------------------------------------------------------------------------------------
// with sh() the rounding to the operand type (bf16 or saturated fp16):
// |q.x - sh(q).sh(x)| = |sh(q).(x - sh(x)) + (q - sh(q)).x|
//                    <= ||sh(q)|| * max||x - sh(x)|| + ||q - sh(q)|| * max||x||      (Cauchy-Schwarz)
// plus a slack for the tensor core's fp32 accumulation: d_pad * 2^-23 * ||sh(q)|| * max||sh(x)||.
__global__ void prep_queries_kernel(const float* __restrict__ q32, __nv_bfloat16* __restrict__ q16,
                                    int nq, int d, int d_pad,
                                    const unsigned int* __restrict__ norm_stats,
                                    float* __restrict__ eps2, float* __restrict__ thr,
                                    int* __restrict__ cnt, int* __restrict__ kept,
                                    int* __restrict__ flags, int sh, int nq_pad,
                                    long long* __restrict__ gstats, int init_cnt,
                                    const DynArgs* __restrict__ dyn) {
    if (dyn) q32 = dyn->q32;
    const int lane = threadIdx.x & 31;
    const int q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (blockIdx.x == 0 && threadIdx.x < GS_COUNT && gstats) gstats[threadIdx.x] = 0;
    if (q >= nq) {
        // rows that pad the last (pair) tile: zeros, so no TMA box hangs over the tensor's end
        if (q < nq_pad) {
            uint2* dst = reinterpret_cast<uint2*>(q16 + static_cast<long long>(q) * d_pad);
            for (int j = lane; j < d_pad / 4; j += 32) dst[j] = make_uint2(0u, 0u);
        }
        return;
    }
    const float4* src = reinterpret_cast<const float4*>(q32 + static_cast<long long>(q) * d);
    uint2* dst = reinterpret_cast<uint2*>(q16 + static_cast<long long>(q) * d_pad);
    float nh = 0.f, nd = 0.f;
    for (int j = lane; j < d_pad / 4; j += 32) {
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (j < d / 4) v = __ldg(src + j);
        uint2 o;
        o.x = pack2_sh(v.x, v.y, sh);
        o.y = pack2_sh(v.z, v.w, sh);
        const float2 flo = unpack2_sh(o.x, sh), fhi = unpack2_sh(o.y, sh);
        const float e0 = v.x - flo.x, e1 = v.y - flo.y, e2 = v.z - fhi.x, e3 = v.w - fhi.y;
        nh += flo.x * flo.x + flo.y * flo.y + fhi.x * fhi.x + fhi.y * fhi.y;
        nd += e0 * e0 + e1 * e1 + e2 * e2 + e3 * e3;
        dst[j] = o;
    }
    nh = warp_sum(nh);
    nd = warp_sum(nd);
    if (lane == 0) {
        const float nx = sqrtf(__uint_as_float(norm_stats[0]));
        const float dx = sqrtf(__uint_as_float(norm_stats[1]));
        const float qh = sqrtf(nh), dq = sqrtf(nd);
        const float acc = static_cast<float>(d_pad) * 1.1920929e-7f;   // d_pad * 2^-23
        float e = qh * dx + dq * nx + acc * qh * (nx + dx);
        e = e * 1.001f + FLT_MIN;          // norms above were themselves rounded
        // no usable bound (overflowing norms, inf in the query): admit everything; the query
        // then overflows its list and is answered by the exact path
        if (!(e <= FLT_MAX)) e = INFINITY;
        eps2[q] = 2.f * e;
        thr[q] = -INFINITY;
        cnt[q] = init_cnt;                 // rows of the dense first slab (stored without counters)
        kept[q] = 0;
        flags[q] = 0;
    }
}

// ---------------------------------------------------------------------------------------
// block-wide radix select
// ---------------------------------------------------------------------------------------
// Top `n_bytes` bytes of the k-th largest of keys[0..n) (1 <= k <= n); low bytes are zero.
// With n_bytes = 4 that is the k-th largest SCORE, with 8 the k-th largest key.
// A threshold only needs a LOWER BOUND of the k-th score: n_bytes = 3 fixes sign, exponent and 15
// mantissa bits (the bound is at most 2^-15 relative below the true value, ~1/500 of the error
// margin it is combined with) and saves a pass.  first_pass / prefix0: leading bytes all keys are
// known to share (see common_prefix_bytes) are not counted again.
__device__ unsigned long long block_radix_select(const unsigned long long* __restrict__ keys,
                                                 int n, int k, int n_bytes, unsigned int* hist,
                                                 unsigned long long* s_prefix, int* s_krem,
                                                 int first_pass = 0, unsigned long long prefix0 = 0ull) {
    const int tid = threadIdx.x, nt = blockDim.x;
    unsigned long long prefix = prefix0;
    int krem = k;
    for (int pass = first_pass; pass < n_bytes; pass++) {
        const int shift = 56 - 8 * pass;
        for (int i = tid; i < 256; i += nt) hist[i] = 0;
        __syncthreads();
        const unsigned long long mask = pass == 0 ? 0ull : (~0ull << (shift + 8));
        // Scores of one list share their leading bytes, so most lanes of a warp hit the SAME bin:
        // lanes with equal digits elect one of them to add the whole group's count.
        for (int base = 0; base < n; base += nt) {
            const int i = base + tid;
            unsigned int digit = 256u;                       // 256 = not counted
            if (i < n) {
                const unsigned long long key = keys[i];
                if ((key & mask) == prefix) digit = static_cast<unsigned int>((key >> shift) & 255);
            }
            // cheap aggregation for the common case: everyone who agrees with lane 0's digit is
            // counted by lane 0 in one add, the rest add for themselves
            const unsigned int first = __shfl_sync(0xffffffffu, digit, 0);
            const unsigned int same = __ballot_sync(0xffffffffu, digit == first);
            if ((tid & 31) == 0) {
                if (digit < 256u) atomicAdd(&hist[digit], static_cast<unsigned int>(__popc(same)));
            } else if (digit < 256u && digit != first) {
                atomicAdd(&hist[digit], 1u);
            }
        }
        __syncthreads();
        if (tid < 32) {
            const int lane = tid;
            unsigned int c[8], sum = 0;
#pragma unroll
            for (int j = 0; j < 8; j++) { c[j] = hist[255 - (8 * lane + j)]; sum += c[j]; }
            unsigned int incl = sum;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned int t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += t;
            }
            const unsigned int excl = incl - sum;
            if (excl < static_cast<unsigned int>(krem) && static_cast<unsigned int>(krem) <= incl) {
                unsigned int r = krem - excl;
                int digit = 0;
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    if (r <= c[j]) { digit = 255 - (8 * lane + j); break; }
                    r -= c[j];
                }
                *s_prefix = prefix | (static_cast<unsigned long long>(digit) << shift);
                *s_krem = static_cast<int>(r);
            }
        }
        __syncthreads();
        prefix = *s_prefix;
        krem = *s_krem;
    }
    return prefix;
}

// LOWER BOUND of the k-th largest score word (high 32 bits) of skeys[0..n) in shared memory, for
// 1 <= k <= n, given the smallest / largest score word of the list (kmin / kmax).  A threshold
// needs no more than a lower bound, so instead of a byte-wise radix select (3 passes over the
// list, each with its own scan) this takes ONE histogram pass of BOUND_BINS equal-width bins over
// [kmin, kmax] -- the scores of a candidate list lie in a narrow range, so a bin is a few thousand
// ulps wide -- and one cheap pass that splits the bin holding the k-th score into 256: the result
// is within 2^(shift-8) key units (typically 32 ulps, 1e-6 relative) below the true value.
// hist: BOUND_BINS words.  Ends with a barrier; s_prefix / s_krem / s_warp are free afterwards.
// K = u64 keys (score word on top) or bare u32 score words; entries whose score word is below kmin
// are not counted (bootstrap_threshold_kernel: empty groups hold 0), so k counts the others.
// Written for a block of 128 or 256 threads; every caller runs SEL_THREADS = 256.
constexpr int BOUND_BINS = 1024;

__device__ __forceinline__ uint32_t score_word(unsigned long long key) { return static_cast<uint32_t>(key >> 32); }
__device__ __forceinline__ uint32_t score_word(uint32_t word) { return word; }

template <class K = unsigned long long>
__device__ uint32_t block_bound_select(const K* skeys, int n, int k, uint32_t kmin,
                                       uint32_t kmax, unsigned int* hist,
                                       unsigned long long* s_prefix, int* s_krem, int* s_warp) {
    if (kmin == kmax) return kmin;
    const uint32_t range = kmax - kmin;
    const int shift = max(0, 32 - __clz(static_cast<int>(range)) - 10);     // (range >> shift) < BOUND_BINS
    const int tid = threadIdx.x, nt = blockDim.x;
    const int lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < BOUND_BINS; i += nt) hist[i] = 0;
    __syncthreads();
    for (int i = tid; i < n; i += nt) {
        const uint32_t hi = score_word(skeys[i]);
        if (hi >= kmin) atomicAdd(&hist[(hi - kmin) >> shift], 1u);
    }
    __syncthreads();
    // thread t owns the `per` bins just below BOUND_BINS - per * t: the top bins come first
    const int per = BOUND_BINS / nt;                     // 4 (SEL_THREADS = 256) or 8 (128 threads)
    const int top = BOUND_BINS - 1 - per * tid;
    unsigned int c[8], sum = 0;
#pragma unroll
    for (int j = 0; j < 8; j++) {
        c[j] = j < per ? hist[top - j] : 0u;
        sum += c[j];
    }
    unsigned int incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) s_warp[warp] = static_cast<int>(incl);
    __syncthreads();
    for (int w = 0; w < warp; w++) incl += static_cast<unsigned int>(s_warp[w]);
    const unsigned int excl = incl - sum;
    if (excl < static_cast<unsigned int>(k) && static_cast<unsigned int>(k) <= incl) {
        unsigned int r = static_cast<unsigned int>(k) - excl;
        int bin = top;
#pragma unroll
        for (int j = 0; j < 8; j++) {
            if (r <= c[j]) { bin = top - j; break; }
            r -= c[j];
        }
        *s_prefix = static_cast<unsigned long long>(bin);
        *s_krem = static_cast<int>(r);
    }
    for (int i = tid; i < 256; i += nt) hist[i] = 0;     // (every thread has read its bins)
    __syncthreads();
    const int bin = static_cast<int>(*s_prefix);
    const int krem = *s_krem;
    uint32_t bound = kmin + (static_cast<uint32_t>(bin) << shift);
    if (shift == 0) { __syncthreads(); return bound; }
    // split that bin into 256 (or 2^shift) sub-bins
    const int sub_shift = max(0, shift - 8);
    for (int i = tid; i < n; i += nt) {
        const uint32_t w = score_word(skeys[i]);
        const uint32_t off = w - kmin;
        if (w >= kmin && static_cast<int>(off >> shift) == bin)
            atomicAdd(&hist[(off - (static_cast<uint32_t>(bin) << shift)) >> sub_shift], 1u);
    }
    __syncthreads();
    if (tid < 32) {
        unsigned int d[8], dsum = 0;
#pragma unroll
        for (int j = 0; j < 8; j++) { d[j] = hist[255 - (8 * lane + j)]; dsum += d[j]; }
        unsigned int dincl = dsum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned int t = __shfl_up_sync(0xffffffffu, dincl, o);
            if (lane >= o) dincl += t;
        }
        const unsigned int dexcl = dincl - dsum;
        if (dexcl < static_cast<unsigned int>(krem) && static_cast<unsigned int>(krem) <= dincl) {
            unsigned int r = static_cast<unsigned int>(krem) - dexcl;
            int digit = 0;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                if (r <= d[j]) { digit = 255 - (8 * lane + j); break; }
                r -= d[j];
            }
            s_warp[0] = digit;
        }
    }
    __syncthreads();
    bound += static_cast<uint32_t>(s_warp[0]) << sub_shift;
    __syncthreads();                                     // s_warp is free again
    return bound;
}

// In-place stream compaction of keys[0..n): keeps keys whose high word is > hi_thr
// (or, with by_key, keys >= key_thr).  Returns the number kept (all threads).
__device__ int block_compact(const unsigned long long* keys, int n, bool by_key, uint32_t hi_thr,
                             unsigned long long key_thr, unsigned long long* out, int* s_warp) {
    const int tid = threadIdx.x, nt = blockDim.x;
    const int lane = tid & 31, warp = tid >> 5, nw = nt >> 5;
    int base_out = 0;
    for (int base = 0; base < n; base += nt) {
        const int i = base + tid;
        unsigned long long key = 0;
        bool keep = false;
        if (i < n) {
            key = keys[i];
            keep = by_key ? (key >= key_thr) : (static_cast<uint32_t>(key >> 32) > hi_thr);
        }
        const unsigned int ballot = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) s_warp[warp] = __popc(ballot);
        __syncthreads();
        int off = 0, tot = 0;
        for (int w = 0; w < nw; w++) {
            const int c = s_warp[w];
            if (w < warp) off += c;
            tot += c;
        }
        if (keep) out[base_out + off + __popc(ballot & ((1u << lane) - 1u))] = key;
        base_out += tot;
        __syncthreads();
    }
    return base_out;
}

// Same selection, for `out` NOT aliasing `keys`: each warp owns a contiguous segment, one
// counting pass, one block barrier, one writing pass (2 barriers instead of 2 per 256 keys).
__device__ int block_compact_disjoint(const unsigned long long* keys, int n, bool by_key,
                                      uint32_t hi_thr, unsigned long long key_thr,
                                      unsigned long long* out, int* s_warp, bool invert = false) {
    const int tid = threadIdx.x, nt = blockDim.x;
    const int lane = tid & 31, warp = tid >> 5, nw = nt >> 5;
    const int seg = ((n + nw - 1) / nw + 31) & ~31;
    const int b = warp * seg, e = min(n, b + seg);
    int mine = 0;
    for (int i0 = b; i0 < e; i0 += 32) {
        const int i = i0 + lane;
        bool keep = false;
        if (i < e) {
            const unsigned long long key = keys[i];
            keep = by_key ? (key >= key_thr) : (static_cast<uint32_t>(key >> 32) > hi_thr);
            keep = keep != invert;
        }
        mine += __popc(__ballot_sync(0xffffffffu, keep));
    }
    if (lane == 0) s_warp[warp] = mine;
    __syncthreads();
    int off = 0, tot = 0;
    for (int w = 0; w < nw; w++) {
        const int c = s_warp[w];
        if (w < warp) off += c;
        tot += c;
    }
    for (int i0 = b; i0 < e; i0 += 32) {
        const int i = i0 + lane;
        unsigned long long key = 0;
        bool keep = false;
        if (i < e) {
            key = keys[i];
            keep = by_key ? (key >= key_thr) : (static_cast<uint32_t>(key >> 32) > hi_thr);
            keep = keep != invert;
        }
        const unsigned int ballot = __ballot_sync(0xffffffffu, keep);
        if (keep) out[off + __popc(ballot & ((1u << lane) - 1u))] = key;
        off += __popc(ballot);
    }
    __syncthreads();
    return tot;
}

// ---------------------------------------------------------------------------------------
// threshold refresh after a slab: one CTA per query
// ---------------------------------------------------------------------------------------
// Let c_k be the k-th largest COARSE score seen so far.  k rows have exact score >= c_k - eps,
// so every member of the final exact top-k has exact >= c_k - eps and coarse >= c_k - 2 eps:
// rows below that can be dropped for good, and later slabs only need to report above it.
// Returns the number of entries the list holds afterwards (block-uniform), or -1 when the query
// overflowed its list (flagged for the exact path).  `scratch` = REFRESH_SMEM_KEYS keys of
// shared memory: lists that fit are pulled into it once, so the select passes and the
// compaction never touch L2 again.
__device__ int refresh_list(int q, int k, int cap, unsigned long long* __restrict__ cand,
                            int* __restrict__ cnt, int* __restrict__ kept, float* __restrict__ thr,
                            const float* __restrict__ eps2, int* __restrict__ flags,
                            long long* __restrict__ gstats, unsigned long long* scratch,
                            unsigned int* hist, unsigned long long* s_prefix, int* s_krem,
                            int* s_warp) {
    const int n = cnt[q];
    const int prev = kept[q];
    const int tid = threadIdx.x;
    if (tid == 0) { s_warp[0] = -1; s_warp[1] = 0; }   // min / max of the staged keys' score words
    __syncthreads();                                 // everyone has read the counters
    if (n > cap) {
        // more hits than the list holds: this query is re-run on the exact path
        if (tid == 0) {
            flags[q] |= FLAG_OVERFLOW;
            thr[q] = INFINITY;
            cnt[q] = 0;
            kept[q] = 0;
            atomicAdd(reinterpret_cast<unsigned long long*>(gstats + GS_OVERFLOW), 1ull);
        }
        return -1;
    }
    if (n == prev) return n;
    if (tid == 0)
        atomicAdd(reinterpret_cast<unsigned long long*>(gstats + GS_CANDIDATES),
                  static_cast<unsigned long long>(n - prev));
    if (n < k) {
        if (tid == 0) kept[q] = n;
        return n;
    }
    unsigned long long* keys = cand + static_cast<long long>(q) * cap;
    const unsigned long long* src = keys;
    uint32_t ck_word;
    if (n <= REFRESH_SMEM_KEYS) {
        // the list is staged in shared memory once; its smallest / largest score word, found on the
        // way, span the histogram of the bound select
        unsigned int lo = 0xFFFFFFFFu, hi = 0u;
        int i = tid;
        const int nt = blockDim.x;
        // four independent loads in flight per thread: this pass is what the kernel waits for
        for (; i + 3 * nt < n; i += 4 * nt) {
            const unsigned long long k0 = keys[i], k1 = keys[i + nt], k2 = keys[i + 2 * nt], k3 = keys[i + 3 * nt];
            scratch[i] = k0; scratch[i + nt] = k1; scratch[i + 2 * nt] = k2; scratch[i + 3 * nt] = k3;
            const unsigned int h0 = static_cast<unsigned int>(k0 >> 32), h1 = static_cast<unsigned int>(k1 >> 32),
                               h2 = static_cast<unsigned int>(k2 >> 32), h3 = static_cast<unsigned int>(k3 >> 32);
            lo = min(min(lo, h0), min(min(h1, h2), h3));
            hi = max(max(hi, h0), max(max(h1, h2), h3));
        }
        for (; i < n; i += nt) {
            const unsigned long long key = keys[i];
            scratch[i] = key;
            lo = min(lo, static_cast<unsigned int>(key >> 32));
            hi = max(hi, static_cast<unsigned int>(key >> 32));
        }
        lo = __reduce_min_sync(0xffffffffu, lo);
        hi = __reduce_max_sync(0xffffffffu, hi);
        if ((tid & 31) == 0) {
            atomicMin(reinterpret_cast<unsigned int*>(&s_warp[0]), lo);
            atomicMax(reinterpret_cast<unsigned int*>(&s_warp[1]), hi);
        }
        __syncthreads();
        src = scratch;
        const unsigned int kmin = static_cast<unsigned int>(s_warp[0]), kmax = static_cast<unsigned int>(s_warp[1]);
        __syncthreads();                             // s_warp is reused by the select and the compaction
        ck_word = block_bound_select(scratch, n, k, kmin, kmax, hist, s_prefix, s_krem, s_warp);
    } else {
        // lists beyond the staging area (k > 1024): 3-byte radix select out of L2
        ck_word = static_cast<uint32_t>(block_radix_select(src, n, k, 3, hist, s_prefix, s_krem) >> 32);
    }
    const float ck = unorder_f32(ck_word);
    float t = __fsub_rd(ck, eps2[q]);
    if (!(t == t)) t = -INFINITY;                    // inf - inf: no usable threshold
    t = nextafterf(t, -INFINITY);                    // admission test is strict
    const int m = (src == keys) ? block_compact(src, n, false, order_f32(t), 0ull, keys, s_warp)
                                : block_compact_disjoint(src, n, false, order_f32(t), 0ull, keys, s_warp);
    if (tid == 0) {
        cnt[q] = m;
        kept[q] = m;
        thr[q] = t;
        atomicMax(reinterpret_cast<unsigned long long*>(gstats + GS_MAX_KEPT),
                  static_cast<unsigned long long>(m));
    }
    return m;
}

// Global threshold of the row-sharded search (peer-direct exchange): after its last slab every
// rank publishes, per query, its m-th largest coarse score with m = ceil(k / world) -- into the
// threshold buffer of EVERY rank (NVLink P2P stores).  On each rank at least m rows score >= its
// own bound, so world * m >= k rows of the whole corpus score >= T = min over ranks: T is a lower
// bound on the global k-th coarse score, and rows with coarse < T - 2 eps cannot be in the global
// exact top-k.  A rank holding fewer than m candidates publishes -inf (no bound).
struct PublishBound {
    int m_rank;                       // 0 = nothing to publish
    int n_dst;
    float* dst[MAX_PEERS];            // dst[i][q]: this rank's row of rank i's threshold buffer
};

__global__ void __launch_bounds__(SEL_THREADS)
refresh_threshold_kernel(int k, int cap, unsigned long long* __restrict__ cand,
                         int* __restrict__ cnt, int* __restrict__ kept, float* __restrict__ thr,
                         const float* __restrict__ eps2, int* __restrict__ flags,
                         long long* __restrict__ gstats, const PublishBound pub) {
    __shared__ unsigned int hist[BOUND_BINS];
    __shared__ unsigned long long s_prefix;
    __shared__ int s_krem;
    __shared__ int s_warp[SEL_THREADS / 32];
    __shared__ unsigned long long skeys[REFRESH_SMEM_KEYS];
    const int q = blockIdx.x;
    int n = -1;
    if (!(flags[q] & FLAG_OVERFLOW))
        n = refresh_list(q, k, cap, cand, cnt, kept, thr, eps2, flags, gstats, skeys, hist, &s_prefix,
                         &s_krem, s_warp);
    if (pub.m_rank > 0) {
        float bound = -INFINITY;
        if (n >= pub.m_rank) {
            __syncthreads();                         // the compacted list is visible to every warp
            const unsigned long long pk = block_radix_select(cand + static_cast<long long>(q) * cap, n,
                                                             pub.m_rank, 3, hist, &s_prefix, &s_krem);
            if ((pk >> 32) != 0ull) bound = unorder_f32(static_cast<uint32_t>(pk >> 32));   // 0 = a NaN score
        }
        if (threadIdx.x < pub.n_dst) pub.dst[threadIdx.x][q] = bound;
    }
}

// Threshold bootstrap of a small batch (tensor_search, latency regime): gmax[q][0..groups) are the
// group maxima (ordered score words, 0 = empty group / NaN) the streaming kernel's group-max launch
// wrote; the k-th largest of them is a lower bound of the query's k-th best coarse score (disjoint
// groups), so thr[q] = that bound - 2 eps_q, exactly what refresh_list derives from a candidate
// list.  Fewer than k non-empty groups: the threshold stays -inf (every row is admitted, the list
// overflows and the query is answered by the exact path).  Dynamic shared memory: groups words.
//
// k <= BOOT_FAST_K (the latency regime's k = 10): no histogram over 19k words.  Each thread keeps
// the maximum of the words it stages; the k-th largest of those 256 thread maxima (rank by
// counting) is itself a lower bound L0 of the k-th largest word -- disjoint subsets again -- and
// only the handful of words >= L0 can be the k-th largest: they are compacted and ranked exactly.
constexpr int BOOT_FAST_K = 64;

__global__ void __launch_bounds__(SEL_THREADS)
bootstrap_threshold_kernel(const uint32_t* __restrict__ gmax, int groups, int k,
                           float* __restrict__ thr, const float* __restrict__ eps2) {
    extern __shared__ uint32_t s_gmax[];
    __shared__ __align__(16) unsigned int hist[BOUND_BINS];   // fast path: thread maxima, then the shortlist
    __shared__ unsigned long long s_prefix;
    __shared__ int s_krem;
    __shared__ int s_warp[SEL_THREADS / 32];
    __shared__ unsigned int s_lo, s_hi, s_valid, s_l0, s_m, s_kth;
    const int q = blockIdx.x;
    const int tid = threadIdx.x;
    if (tid == 0) { s_lo = 0xFFFFFFFFu; s_hi = 0u; s_valid = 0u; s_l0 = 0xFFFFFFFFu; s_m = 0u; s_kth = 0u; }
    const uint4* src = reinterpret_cast<const uint4*>(gmax + static_cast<long long>(q) * groups);   // groups % 128 == 0
    // the staging pass is what this kernel waits for: every load of a thread in flight at once
    // (BOOT_MAX_GROUPS / 4 / SEL_THREADS = 20 uint4 per thread at most)
    constexpr int kPerThread = BOOT_MAX_GROUPS / 4 / SEL_THREADS;
    uint4 v[kPerThread];
#pragma unroll
    for (int j = 0; j < kPerThread; j++) {
        const int i = tid + j * SEL_THREADS;
        v[j] = src[min(i, groups / 4 - 1)];       // unpredicated (7 predicate registers would cap the loads in flight)
    }
    unsigned int my_max = 0u;
#pragma unroll
    for (int j = 0; j < kPerThread; j++) {
        const int i = tid + j * SEL_THREADS;
        if (i < groups / 4) {
            reinterpret_cast<uint4*>(s_gmax)[i] = v[j];
            my_max = max(max(my_max, max(v[j].x, v[j].y)), max(v[j].z, v[j].w));
        }
    }
    hist[tid] = my_max;
    __syncthreads();
    uint32_t ck_word = 0u;
    bool have = false;
    if (k <= BOOT_FAST_K) {
        // r = how many thread maxima are strictly greater than mine.  The k-th largest of the 256
        // is the smallest one with r <= k - 1 (ties share their r): L0.  Threads without a word hold
        // 0; fewer than k non-empty threads -> L0 = 0 and the general path below takes over.
        int r = 0;
        const uint4* h4 = reinterpret_cast<const uint4*>(hist);
#pragma unroll 4
        for (int j = 0; j < SEL_THREADS / 4; j++) {
            const uint4 o = h4[j];
            r += (o.x > my_max ? 1 : 0) + (o.y > my_max ? 1 : 0) + (o.z > my_max ? 1 : 0) + (o.w > my_max ? 1 : 0);
        }
        if (r <= k - 1) atomicMin(&s_l0, my_max);
        __syncthreads();
        const unsigned int l0 = s_l0;
        if (l0 != 0u) {
            unsigned int* shortlist = hist + SEL_THREADS;        // BOUND_BINS - SEL_THREADS words
            for (int i = tid; i < groups / 4; i += SEL_THREADS) {
                const uint4 w4 = reinterpret_cast<const uint4*>(s_gmax)[i];
                const unsigned int w[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
                for (int j = 0; j < 4; j++)
                    if (w[j] >= l0) {
                        const unsigned int pos = atomicAdd(&s_m, 1u);
                        if (pos < static_cast<unsigned int>(BOUND_BINS - SEL_THREADS)) shortlist[pos] = w[j];
                    }
            }
            __syncthreads();
            const int m = static_cast<int>(s_m);                 // >= k: k thread maxima are >= L0
            if (m <= BOUND_BINS - SEL_THREADS) {
                // exact k-th largest of the shortlist: element i has rank = #(greater) + #(equal before it)
                for (int i = tid; i < m; i += SEL_THREADS) {
                    const unsigned int mine = shortlist[i];
                    int rk = 0;
                    for (int j = 0; j < m; j++) {
                        const unsigned int o = shortlist[j];
                        rk += (o > mine || (o == mine && j < i)) ? 1 : 0;
                    }
                    if (rk == k - 1) s_kth = mine;
                }
                __syncthreads();
                ck_word = s_kth;
                have = true;
            }
        }
        __syncthreads();                                     // hist is reused below
    }
    if (!have) {
        // general path (k > BOOT_FAST_K, empty groups / NaN scores, thousands of ties): smallest /
        // largest non-empty word and their count, then the histogram bound select.  The group maxima
        // span a wide range (all of [min score, max score], not a candidate list's narrow top): a
        // second select over [first bound, max] brings the bound within a few ulps of the k-th
        unsigned int lo = 0xFFFFFFFFu, hi = 0u, valid = 0u;
        for (int i = tid; i < groups; i += SEL_THREADS) {
            const unsigned int w = s_gmax[i];
            if (w != 0u) { lo = min(lo, w); hi = max(hi, w); valid++; }
        }
        lo = __reduce_min_sync(0xffffffffu, lo);
        hi = __reduce_max_sync(0xffffffffu, hi);
        valid = __reduce_add_sync(0xffffffffu, valid);
        if ((tid & 31) == 0) {
            atomicMin(&s_lo, lo);
            atomicMax(&s_hi, hi);
            atomicAdd(&s_valid, valid);
        }
        __syncthreads();
        if (static_cast<int>(s_valid) < k) return;           // thr[q] stays -inf (prep_queries_kernel)
        const unsigned int kmin = s_lo, kmax = s_hi;
        __syncthreads();
        ck_word = block_bound_select<uint32_t>(s_gmax, groups, k, kmin, kmax, hist,
                                               &s_prefix, &s_krem, s_warp);
        ck_word = block_bound_select<uint32_t>(s_gmax, groups, k, ck_word, kmax, hist,
                                               &s_prefix, &s_krem, s_warp);
    }
    if (tid == 0) {
        float t = __fsub_rd(unorder_f32(ck_word), eps2[q]);
        if (!(t == t)) t = -INFINITY;                        // inf - inf: no usable threshold
        thr[q] = nextafterf(t, -INFINITY);                   // admission test is strict
    }
}

__global__ void fill_float_kernel(float* dst, long long count, float v) {
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < count;
         i += static_cast<long long>(gridDim.x) * blockDim.x)
        dst[i] = v;
}

// ---------------------------------------------------------------------------------------
// finalize: (optional) fp32 rescore of the surviving candidates, exact top-k, sorted output
// ---------------------------------------------------------------------------------------
struct FinalizeParams {
    int k, cap, d;
    const int* qlist;                 // slot -> query index (nullptr: identity)
    unsigned long long* cand;         // [slots, cap]
    const int* cnt;                   // [slots] entries per slot
    const int* flags;                 // [slots] or nullptr
    // fused last threshold refresh (tensor path; nullptr otherwise): the raw fill counters, the
    // kept counts, thresholds, bounds and flags the refresh kernel would have updated
    int* r_cnt; int* r_kept; float* r_thr; const float* r_eps2; int* r_flags;
    const float* eps2;                // [slots] 2*eps per query: enables the two-stage rescore
    const float* cert_eps2;           // [slots] 2*eps per query: run-time check |coarse - exact| <= eps (or nullptr)
    const float* q32;                 // [*, d] fp32 queries (rescore)
    const float* x32;                 // [n, d] fp32 corpus (rescore), or nullptr:
    const __nv_bfloat16* x16;         // [n, d_pad] 16-bit corpus when the index stores bf16 / fp16
    int d_pad;
    int sh;                           // SH_BF16 / SH_F16: element type of x16
    long long row_offset;             // reported id = local row + row_offset, or (n_seg > 0):
    int n_seg;                        // local row + seg_delta[s], s = last segment with
    const long long* seg_local;       // seg_local[s] <= local row (shards made of several
    const long long* seg_delta;       // global row ranges)
    float* out_scores;                // [*, k]
    long long* out_rows;              // [*, k]
    // peer-direct exchange: the same results are also stored into these buffers, which live in
    // the OTHER GPUs' memory (NVLink P2P stores), so no separate all-gather is needed
    int n_extra;
    float* extra_s[MAX_PEERS - 1];
    long long* extra_r[MAX_PEERS - 1];
    // owner mode (owner_per > 0): query q of the search belongs to rank q / owner_per and its block
    // is stored ONLY there (locally when that is self_rank, else into extra slot e with
    // extra_rank[e] == owner): 1/world of the peer traffic, and the merge of a query runs once
    int owner_per, self_rank;
    int extra_rank[MAX_PEERS - 1];
    long long q_base;                 // index of slot 0 in the whole search (query batches)
    // global threshold round (g_thr != nullptr): wait for every rank's bound, prune with the minimum
    const float* g_thr;               // [g_world, g_stride] this rank's threshold buffer
    const unsigned int* g_flags;      // this rank's flag array of the parity
    int g_world;
    long long g_stride;
    unsigned int g_seq;
    long long g_timeout_ns;
    long long* gstats;
    int ring_stages;                  // rescore: rows in flight per warp (1-D TMA ring in shared memory)
    const DynArgs* dyn;               // graph replay: q32 / g_seq (and, with dyn_out, the output buffers) come from here
    int dyn_out;
};

__device__ void block_bitonic_desc(unsigned long long* s, int P) {
    for (int size = 2; size <= P; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int i = threadIdx.x; i < P / 2; i += blockDim.x) {
                const int lo = 2 * i - (i & (stride - 1));
                const int hi = lo + stride;
                const bool desc = (lo & size) == 0;
                const unsigned long long a = s[lo], b = s[hi];
                if ((a < b) == desc) { s[lo] = b; s[hi] = a; }
            }
            __syncthreads();
        }
    }
}

// kRows = how the rows the rescore reads are stored: ROWS_F32 (fp32 master rows, p.x32) or
// ROWS_BF16 / ROWS_F16 (a 16-bit store, p.x16) -- a compile-time constant, so the inner loop of the
// rescore (instruction-issue bound) carries one unpack sequence instead of both under predicates.
enum { ROWS_F32 = 0, ROWS_BF16 = 1, ROWS_F16 = 2 };

template <bool kRescore, int kRows = ROWS_F32>
__global__ void __launch_bounds__(SEL_THREADS, 3) finalize_kernel(const __grid_constant__ FinalizeParams p) {
    // graph replay: the per-call values come from DynArgs (the parameter block itself stays in
    // constant memory: no local copy)
    const float* const q32 = p.dyn ? p.dyn->q32 : p.q32;
    const unsigned int g_seq = p.dyn ? p.dyn->seq : p.g_seq;
    float* const out_scores = (p.dyn && p.dyn_out) ? p.dyn->out_s : p.out_scores;
    long long* const out_rows = (p.dyn && p.dyn_out) ? p.dyn->out_r : p.out_rows;
    extern __shared__ __align__(16) uint8_t fsm[];
    unsigned long long* sbuf = reinterpret_cast<unsigned long long*>(fsm);   // [SORT_CAP]
    // dynamic shared memory: [sort buffer, aliased by the rescore's row ring | query fp32 [d] | ring mbarriers]
    // (the ring is live only inside rescore_range, the sort buffer only outside of it)
    const size_t union_bytes = kRescore ? max(static_cast<size_t>(SORT_CAP) * sizeof(unsigned long long),
                                              static_cast<size_t>(blockDim.x >> 5) * p.ring_stages *
                                                  (kRows == ROWS_F32 ? static_cast<size_t>(p.d) * 4 : static_cast<size_t>(p.d_pad) * 2))
                                        : static_cast<size_t>(SORT_CAP) * sizeof(unsigned long long);
    float* sq = reinterpret_cast<float*>(fsm + union_bytes);                             // the query, [d] fp32
    __shared__ unsigned int hist[BOUND_BINS];     // (the fused refresh's bound select needs all of it)
    __shared__ unsigned long long s_prefix;
    __shared__ int s_krem;
    __shared__ int s_warp[SEL_THREADS / 32];
    __shared__ unsigned int s_min;
    __shared__ unsigned int s_err;      // max |coarse - exact| / eps of this query (float bits, >= 0)
    __shared__ unsigned int s_viol;

    const int slot = blockIdx.x;
    if (p.flags && (p.flags[slot] & FLAG_OVERFLOW)) return;
    const int q = p.qlist ? p.qlist[slot] : slot;
    int n;
    if (kRescore && p.r_cnt) {
        // the refresh that would follow the last slab, done here: one launch and one pass over
        // the list less (sbuf doubles as its staging area: SORT_CAP == REFRESH_SMEM_KEYS)
        n = refresh_list(slot, p.k, p.cap, p.cand, p.r_cnt, p.r_kept, p.r_thr, p.r_eps2, p.r_flags,
                         p.gstats, sbuf, hist, &s_prefix, &s_krem, s_warp);
        if (n < 0) return;
        __syncthreads();                             // compacted list visible to every warp
    } else {
        n = min(p.cnt[slot], p.cap);
    }
    unsigned long long* keys = p.cand + static_cast<long long>(slot) * p.cap;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;

    if (kRescore && p.g_thr) {
        // row-sharded search: every rank's bound for this query is (about to be) in my threshold
        // buffer; T = their minimum bounds the GLOBAL k-th coarse score from below (PublishBound)
        wait_peer_flags(p.g_flags, p.g_world, XF_THR, g_seq, p.g_timeout_ns,
                        p.gstats ? p.gstats + GS_XSTATUS : nullptr);
        float T = INFINITY;
        for (int r = 0; r < p.g_world; r++) {
            const float b = p.g_thr[r * p.g_stride + p.q_base + slot];
            T = (b == b) ? fminf(T, b) : -INFINITY;
        }
        float tg = __fsub_rd(T, p.cert_eps2[slot]);
        if (!(tg == tg)) tg = -INFINITY;
        tg = nextafterf(tg, -INFINITY);              // kept: coarse > tg
        if (tg > -INFINITY && n > 0) {
            n = block_compact(keys, n, false, order_f32(tg), 0ull, keys, s_warp);
            __syncthreads();
        }
    }

    if (kRescore) {
        if (threadIdx.x == 0) {
            s_err = 0u; s_viol = 0u;
            uint64_t* b0 = reinterpret_cast<uint64_t*>(fsm + union_bytes + ((static_cast<size_t>(p.d) * 4 + 15) & ~static_cast<size_t>(15)));
            for (int i = 0; i < (blockDim.x >> 5) * p.ring_stages; i++) ptx::mbar_init(&b0[i], 1);
            ptx::fence_mbar_init();
        }
        for (int j = threadIdx.x; j < p.d; j += blockDim.x)
            sq[j] = q32[static_cast<long long>(q) * p.d + j];
        __syncthreads();
        // Run-time certificate of the a-priori bound eps_q (prep_queries_kernel): every row that is
        // rescored anyway still carries its COARSE score in the key, so |coarse - exact| / eps_q is
        // free to check.  It is the only guard on the tensor core's fp32 accumulation behaviour.
        const float cert_eps = p.cert_eps2 ? 0.5f * p.cert_eps2[slot] : 0.f;
        const bool cert = p.gstats && cert_eps > 0.f && cert_eps <= FLT_MAX;
        // keys[lo..hi) <- exact (score,row) keys.  track_min: s_min <- smallest exact score (ordered).
        //
        // The rescore is a GATHER: 1.5-3 KB from a random HBM page per surviving row, ~150 (k = 100)
        // to ~1500 (k = 1000) rows per query.  Every row is one contiguous chunk, so it is fetched
        // by ONE 1-D TMA (cp.async.bulk) into a per-warp ring in shared memory: the bytes in flight
        // (ring_stages rows per warp, ~70 KB per CTA) no longer depend on registers or occupancy,
        // and the arithmetic reads the row from shared memory against the query slice each lane
        // keeps in registers for the whole kernel.  Products are summed four at a time in fp32 (3
        // roundings of ~6e-8 relative on a 4-term partial) and the partials accumulated in fp64.
        auto dot4 = [](float4 a, float4 b) {
            float t = a.x * b.x;
            t = fmaf(a.y, b.y, t);
            t = fmaf(a.z, b.z, t);
            return fmaf(a.w, b.w, t);
        };
        constexpr bool rows16 = kRows != ROWS_F32;
        constexpr int kSh = kRows == ROWS_F16 ? SH_F16 : SH_BF16;
        const int chunk_elems = rows16 ? 8 : 4;                    // elements per 16-byte chunk of a stored row
        const int row_bytes = rows16 ? p.d_pad * 2 : p.d * 4;
        const int n_chunks = row_bytes >> 4;
        const char* const row_base = rows16 ? reinterpret_cast<const char*>(p.x16)
                                            : reinterpret_cast<const char*>(p.x32);
        // this lane's slice of the query: chunk c = lane + 32 u covers elements [c*E, c*E + E)
        float4 qreg[RESCORE_JU];
        const bool q_in_regs = p.d <= 128 * RESCORE_JU;
        if (q_in_regs) {
#pragma unroll
            for (int u = 0; u < RESCORE_JU; u++) {
                // fp32 rows: float4 number (lane + 32 u); 16-bit rows: float4 numbers 2c, 2c+1 of chunk c = lane + 32 (u/2)
                const int f4 = rows16 ? 2 * (lane + 32 * (u >> 1)) + (u & 1) : lane + 32 * u;
                qreg[u] = (4 * f4 < p.d) ? reinterpret_cast<const float4*>(sq)[f4] : make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
        auto row_dot = [&](const uint4* srow) -> double {          // all lanes; partial of this lane
            double acc = 0.0;
            if (q_in_regs) {
                if (!rows16) {
#pragma unroll
                    for (int u = 0; u < RESCORE_JU; u++) {
                        const int c = lane + 32 * u;
                        if (c < n_chunks) {
                            const uint4 v = srow[c];
                            acc += static_cast<double>(dot4(make_float4(__uint_as_float(v.x), __uint_as_float(v.y),
                                                                        __uint_as_float(v.z), __uint_as_float(v.w)), qreg[u]));
                        }
                    }
                } else {
#pragma unroll
                    for (int u = 0; u < RESCORE_JU / 2; u++) {
                        const int c = lane + 32 * u;
                        if (c < n_chunks) {
                            const uint4 v = srow[c];
                            const float2 e0 = unpack2_t<kSh>(v.x), e1 = unpack2_t<kSh>(v.y);
                            const float2 e2 = unpack2_t<kSh>(v.z), e3 = unpack2_t<kSh>(v.w);
                            acc += static_cast<double>(dot4(make_float4(e0.x, e0.y, e1.x, e1.y), qreg[2 * u]));
                            acc += static_cast<double>(dot4(make_float4(e2.x, e2.y, e3.x, e3.y), qreg[2 * u + 1]));
                        }
                    }
                }
            } else {                                               // d > 1024: query slice from shared memory
                const float4* q4 = reinterpret_cast<const float4*>(sq);
                for (int c = lane; c < n_chunks; c += 32) {
                    const uint4 v = srow[c];
                    if (!rows16) {
                        acc += static_cast<double>(dot4(make_float4(__uint_as_float(v.x), __uint_as_float(v.y),
                                                                    __uint_as_float(v.z), __uint_as_float(v.w)), q4[c]));
                    } else {
                        const float2 e0 = unpack2_t<kSh>(v.x), e1 = unpack2_t<kSh>(v.y);
                        const float2 e2 = unpack2_t<kSh>(v.z), e3 = unpack2_t<kSh>(v.w);
                        const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
                        const float4 qa = (8 * c < p.d) ? q4[2 * c] : z, qb = (8 * c + 4 < p.d) ? q4[2 * c + 1] : z;
                        acc += static_cast<double>(dot4(make_float4(e0.x, e0.y, e1.x, e1.y), qa));
                        acc += static_cast<double>(dot4(make_float4(e2.x, e2.y, e3.x, e3.y), qb));
                    }
                }
            }
            return acc;
        };
        (void)chunk_elems;
        const int NS = p.ring_stages;
        uint8_t* const ring = fsm;                                 // aliases the sort buffer (see the layout note above)
        uint64_t* const bars = reinterpret_cast<uint64_t*>(fsm + union_bytes + ((static_cast<size_t>(p.d) * 4 + 15) & ~static_cast<size_t>(15)));
        uint8_t* const my_ring = ring + static_cast<size_t>(warp) * NS * row_bytes;
        uint64_t* const my_bars = bars + warp * NS;
        // The per-row epilogue (certificate, key, minimum) is done 32 rows at a time, one row per
        // lane, instead of by lane 0 after every row: the rescore is instruction-issue bound once
        // the gather is asynchronous, and a serial one-lane tail was a third of its instructions.
        const float inv_cert_eps = cert ? 1.0f / cert_eps : 0.f;
        float w_err = 0.f;                 // lane-local maxima / minima, folded into shared memory once per warp
        unsigned int w_viol = 0u, w_min = 0xFFFFFFFFu;
        int st_i = 0, st_w = 0;            // ring stage of the next row to issue / to wait for
        unsigned int ph_w = 0u;            // phase bit of stage st_w
        auto rescore_range = [&](int lo, int hi, bool track_min) {
            const int cnt_w = (hi - lo - warp + nw - 1) / nw;      // rows of this warp: lo + warp + n * nw
            if (cnt_w <= 0) return;
            auto issue = [&](int n) {                              // lane 0: fetch this warp's n-th row
                const uint32_t row = key_row(keys[lo + warp + n * nw]);
                ptx::mbar_expect_tx(&my_bars[st_i], static_cast<uint32_t>(row_bytes));
                ptx::bulk_load(my_ring + static_cast<size_t>(st_i) * row_bytes,
                               row_base + static_cast<size_t>(row) * row_bytes, static_cast<uint32_t>(row_bytes),
                               &my_bars[st_i], ptx::kEvictFirst);
                if (++st_i == NS) st_i = 0;
            };
            if (lane == 0)
                for (int n = 0; n < min(NS, cnt_w); n++) issue(n);
            double mine = 0.0;                                     // total of row (n0 + lane) of the current group of 32
            auto epilogue = [&](int n0, int cnt) {                 // rows n0 .. n0+cnt-1, lane = row - n0
                if (lane < cnt) {
                    const int i = lo + warp + (n0 + lane) * nw;
                    const unsigned long long key1 = keys[i];
                    const float s1 = static_cast<float>(mine);
                    if (cert) {
                        const float e = fabsf(key_score(key1) - s1);
                        if (e <= FLT_MAX) {                        // NaN / inf scores carry no margin (see shadow_rows_kernel)
                            const float ratio = e * inv_cert_eps;
                            w_err = fmaxf(w_err, ratio);
                            w_viol += ratio > 1.0f ? 1u : 0u;
                        }
                    }
                    keys[i] = make_key(s1, key_row(key1));         // NaN -> high word 0
                    if (track_min) w_min = min(w_min, order_f32(s1));   // order(NaN) = 0: no pruning
                }
            };
            for (int n = 0; n < cnt_w; n++) {
                ptx::mbar_wait(&my_bars[st_w], ph_w);
                double acc = row_dot(reinterpret_cast<const uint4*>(my_ring + static_cast<size_t>(st_w) * row_bytes));
                if (++st_w == NS) { st_w = 0; ph_w ^= 1u; }
                __syncwarp();                                      // every lane is done with the stage
                if (lane == 0 && n + NS < cnt_w) issue(n + NS);
                acc = warp_sum(acc);
                if (lane == (n & 31)) mine = acc;
                if ((n & 31) == 31) epilogue(n - 31, 32);
            }
            if (cnt_w & 31) epilogue(cnt_w & ~31, cnt_w & 31);
        };
        auto fold_warp_stats = [&]() {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                w_err = fmaxf(w_err, __shfl_xor_sync(0xffffffffu, w_err, o));
                w_viol += __shfl_xor_sync(0xffffffffu, w_viol, o);
                w_min = min(w_min, __shfl_xor_sync(0xffffffffu, w_min, o));
            }
            if (lane == 0) {
                if (w_err > 0.f) atomicMax(&s_err, __float_as_uint(w_err));
                if (w_viol) atomicAdd(&s_viol, w_viol);
                atomicMin(&s_min, w_min);
            }
            w_min = 0xFFFFFFFFu;
        };
        int n_resc = n;
        if (p.eps2 && n - p.k >= 64 && n <= SORT_CAP) {   // (not worth a select for a handful of rows)
            // Two-stage rescore.  T = the rows holding the k best COARSE scores (ties included):
            // after their exact rescore, k rows are known with exact score >= s' = min over T, so
            // the final k-th exact score is >= s' and a member y of the final top-k has
            // coarse(y) >= exact(y) - eps >= s' - eps: only those of the remaining rows are
            // rescored (the list itself was cut at c_k - 2 eps; this halves the window).
            for (int i = threadIdx.x; i < n; i += blockDim.x) sbuf[i] = keys[i];
            if (threadIdx.x == 0) s_min = 0xFFFFFFFFu;
            __syncthreads();
            // (3 bytes: T is then a superset of the k best coarse scores -- at least k rows, as needed)
            const unsigned long long pk = block_radix_select(sbuf, n, p.k, 3, hist, &s_prefix, &s_krem);
            const int m1 = block_compact_disjoint(sbuf, n, true, 0u, pk, keys, s_warp);            // T
            const int rest = block_compact_disjoint(sbuf, n, true, 0u, pk, keys + m1, s_warp, true);
            ptx::fence_proxy_async_smem();               // sbuf (generic proxy) is about to be overwritten by TMA
            __syncthreads();
            rescore_range(0, m1, true);
            fold_warp_stats();
            __syncthreads();
            const uint32_t omin = s_min;
            float t2 = omin == 0u ? -INFINITY : __fsub_rd(unorder_f32(omin), 0.5f * p.eps2[slot]);
            if (!(t2 == t2)) t2 = -INFINITY;                 // inf - inf: no usable threshold
            t2 = nextafterf(t2, -INFINITY);                  // kept: coarse > t2
            const int m2 = block_compact_disjoint(keys + m1, rest, false, order_f32(t2), 0ull, sbuf, s_warp);
            for (int i = threadIdx.x; i < m2; i += blockDim.x) keys[m1 + i] = sbuf[i];
            ptx::fence_proxy_async_smem();
            __syncthreads();
            rescore_range(m1, m1 + m2, false);
            n_resc = m1 + m2;
        } else {
            ptx::fence_proxy_async_smem();               // (the fused refresh staged the list in sbuf)
            __syncthreads();
            rescore_range(0, n, false);
        }
        fold_warp_stats();
        __syncthreads();
        if (threadIdx.x == 0 && p.gstats) {
            atomicAdd(reinterpret_cast<unsigned long long*>(p.gstats + GS_RESCORED),
                      static_cast<unsigned long long>(n_resc));
            if (s_err) atomicMax(reinterpret_cast<unsigned long long*>(p.gstats + GS_MAX_ERR),
                                 static_cast<unsigned long long>(s_err));
            if (s_viol) atomicAdd(reinterpret_cast<unsigned long long*>(p.gstats + GS_VIOLATIONS),
                                  static_cast<unsigned long long>(s_viol));
        }
        n = n_resc;
    }

    int m;   // entries to sort
    if (n <= SORT_CAP) {
        for (int i = threadIdx.x; i < n; i += blockDim.x) sbuf[i] = keys[i];
        m = n;
    } else {
        // more survivors than the sort buffer: radix-select the k best keys first
        const unsigned long long kth = block_radix_select(keys, n, p.k, 8, hist, &s_prefix, &s_krem);
        m = block_compact_disjoint(keys, n, true, 0u, kth, sbuf, s_warp);
    }
    int P = 1;
    while (P < m) P <<= 1;
    if (P < 2) P = 2;
    for (int i = m + threadIdx.x; i < P; i += blockDim.x) sbuf[i] = 0ull;
    __syncthreads();
    block_bitonic_desc(sbuf, P);
    for (int j = threadIdx.x; j < p.k; j += blockDim.x) {
        float s = -FLT_MAX;
        long long r = -1;
        if (j < m) {
            const unsigned long long key = sbuf[j];
            if ((key >> 32) != 0ull) {
                s = key_score(key);
                r = static_cast<long long>(key_row(key));
                if (p.n_seg > 0) {
                    int lo = 0, hi = p.n_seg - 1;          // last segment starting at or before r
                    while (lo < hi) {
                        const int mid = (lo + hi + 1) >> 1;
                        if (p.seg_local[mid] <= r) lo = mid; else hi = mid - 1;
                    }
                    r += p.seg_delta[lo];
                } else {
                    r += p.row_offset;
                }
            }
        }
        const long long o = static_cast<long long>(q) * p.k + j;
        const int owner = p.owner_per > 0 ? static_cast<int>((p.q_base + q) / p.owner_per) : -1;
        if (owner < 0 || owner == p.self_rank) {
            out_scores[o] = s;
            out_rows[o] = r;
        }
        for (int e = 0; e < p.n_extra; e++) {
            if (owner < 0 || owner == p.extra_rank[e]) {
                p.extra_s[e][o] = s;
                p.extra_r[e][o] = r;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------
// exact path: fp32 FMA scores for up to EXACT_QB queries, then a multi-CTA radix select
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
exact_scores_kernel(const float* __restrict__ x32, const __nv_bfloat16* __restrict__ x16,
                    long long n, int d, int d_pad, int sh, const float* __restrict__ q32, const int* __restrict__ qlist, int nqg,
                    float* __restrict__ scores /*[EXACT_QB, n]*/) {
    extern __shared__ __align__(16) float esq[];   // [EXACT_QB, d]
    for (int i = threadIdx.x; i < EXACT_QB * d; i += blockDim.x) {
        const int b = i / d, j = i - b * d;
        esq[i] = b < nqg ? q32[static_cast<long long>(qlist[b]) * d + j] : 0.f;
    }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const long long warp = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
    const int d4 = d / 4;
    const float4* sq4 = reinterpret_cast<const float4*>(esq);
    for (long long r = warp; r < n; r += nwarps) {
        float acc[EXACT_QB];
#pragma unroll
        for (int b = 0; b < EXACT_QB; b++) acc[b] = 0.f;
        for (int j = lane; j < d4; j += 32) {
            const float4 xv = load_row4(x32, x16, r, d, d_pad, j, sh);
#pragma unroll
            for (int b = 0; b < EXACT_QB; b++) {
                const float4 qv = sq4[b * d4 + j];
                acc[b] = fmaf(xv.x, qv.x, acc[b]);
                acc[b] = fmaf(xv.y, qv.y, acc[b]);
                acc[b] = fmaf(xv.z, qv.z, acc[b]);
                acc[b] = fmaf(xv.w, qv.w, acc[b]);
            }
        }
        float mine = 0.f;
#pragma unroll
        for (int b = 0; b < EXACT_QB; b++) {
            const float s = warp_sum(acc[b]);
            if (lane == b) mine = s;
        }
        if (lane < nqg) scores[static_cast<long long>(lane) * n + r] = mine;
    }
}

// per-query select state of the exact path
struct ExactState {
    unsigned long long prefix[EXACT_QB];
    int krem[EXACT_QB];
    int take_all[EXACT_QB];
};

__global__ void exact_init_kernel(ExactState* st, unsigned int* ghist, int* cnt, int k) {
    const int i = threadIdx.x;
    if (i < EXACT_QB) { st->prefix[i] = 0; st->krem[i] = k; st->take_all[i] = 0; cnt[i] = 0; }
    for (int j = i; j < EXACT_QB * 256; j += blockDim.x) ghist[j] = 0;
}

__global__ void __launch_bounds__(256)
exact_hist_kernel(const float* __restrict__ scores, long long n, int pass,
                  const ExactState* __restrict__ st, unsigned int* __restrict__ ghist) {
    __shared__ unsigned int hist[256];
    const int g = blockIdx.y;
    if (st->take_all[g]) return;
    hist[threadIdx.x] = 0;
    __syncthreads();
    const int shift = 56 - 8 * pass;
    const unsigned long long mask = pass == 0 ? 0ull : (~0ull << (shift + 8));
    const unsigned long long prefix = st->prefix[g];
    const float* s = scores + static_cast<long long>(g) * n;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const unsigned long long key = make_key(s[i], static_cast<uint32_t>(i));
        if ((key >> 32) != 0ull && (key & mask) == prefix)
            atomicAdd(&hist[(key >> shift) & 255], 1u);
    }
    __syncthreads();
    const unsigned int c = hist[threadIdx.x];
    if (c) atomicAdd(&ghist[g * 256 + threadIdx.x], c);
}

__global__ void exact_pick_kernel(ExactState* st, unsigned int* ghist, int pass) {
    const int g = blockIdx.x, lane = threadIdx.x;
    if (st->take_all[g]) return;
    unsigned int* h = ghist + g * 256;
    const int shift = 56 - 8 * pass;
    const int krem = st->krem[g];
    unsigned int c[8], sum = 0;
#pragma unroll
    for (int j = 0; j < 8; j++) { c[j] = h[255 - (8 * lane + j)]; sum += c[j]; }
    unsigned int incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    const unsigned int total = __shfl_sync(0xffffffffu, incl, 31);
    const unsigned int excl = incl - sum;
    __syncwarp();
#pragma unroll
    for (int j = 0; j < 8; j++) h[255 - (8 * lane + j)] = 0;   // ready for the next pass
    if (total < static_cast<unsigned int>(krem)) {
        // fewer than k reportable rows in total: everything is a result
        if (lane == 0) { st->take_all[g] = 1; st->prefix[g] = 0; }
        return;
    }
    if (excl < static_cast<unsigned int>(krem) && static_cast<unsigned int>(krem) <= incl) {
        unsigned int r = krem - excl;
        int digit = 0;
#pragma unroll
        for (int j = 0; j < 8; j++) {
            if (r <= c[j]) { digit = 255 - (8 * lane + j); break; }
            r -= c[j];
        }
        st->prefix[g] |= static_cast<unsigned long long>(digit) << shift;
        st->krem[g] = static_cast<int>(r);
    }
}

__global__ void __launch_bounds__(256)
exact_collect_kernel(const float* __restrict__ scores, long long n, const ExactState* __restrict__ st,
                     unsigned long long* __restrict__ cand, int* __restrict__ cnt, int cap) {
    const int g = blockIdx.y;
    const unsigned long long kth = st->prefix[g];
    const float* s = scores + static_cast<long long>(g) * n;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const unsigned long long key = make_key(s[i], static_cast<uint32_t>(i));
        if ((key >> 32) != 0ull && key >= kth) {
            const int slot = atomicAdd(cnt + g, 1);
            if (slot < cap) cand[static_cast<long long>(g) * cap + slot] = key;
        }
    }
}

// ---------------------------------------------------------------------------------------
// peer-direct exchange: publish "my results for search `seq` are in your memory"
// ---------------------------------------------------------------------------------------
struct PeerFlags {
    int world, rank;
    unsigned int* flags[MAX_PEERS];   // flags[p] = rank p's flag array of this parity, [XF_WORDS * world]
};
// Launched after the kernel whose peer stores it announces, on the same stream: the kernel
// boundary makes those stores (local and peer) performed, the system fence orders them before
// the flag.  word = XF_RESULT (after finalize; also publishes the overflow count) or XF_THR
// (after the last refresh).
__global__ void exchange_signal_kernel(PeerFlags pf, unsigned int seq, int word,
                                       const long long* __restrict__ gstats, long long prior_overflow,
                                       const DynArgs* __restrict__ dyn) {
    if (dyn) seq = dyn->seq;
    const int p = threadIdx.x;
    if (p >= pf.world) return;
    unsigned int* f = pf.flags[p] + XF_WORDS * pf.rank;
    if (word == XF_RESULT) {
        const long long ov = gstats[GS_OVERFLOW] + prior_overflow;
        f[XF_OVERFLOW] = ov > 0x7fffffffll ? 0x7fffffffu : static_cast<unsigned int>(ov);
    }
    __threadfence_system();
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(f + word), "r"(seq) : "memory");
}

// A rank that owns no query of a search (owner mode, nq < world) has nothing to merge but still
// reports the exchange status (overflows, timeouts) like everyone else.
__global__ void exchange_wait_kernel(const unsigned int* wait_flags, int world, unsigned int seq,
                                     long long* __restrict__ xstatus, long long timeout_ns,
                                     const DynArgs* __restrict__ dyn) {
    if (dyn) seq = dyn->seq;
    wait_peer_flags(wait_flags, world, XF_RESULT, seq, timeout_ns, xstatus);
    if (threadIdx.x == 0) {
        long long ov = 0;
        for (int l = 0; l < world; l++) ov += wait_flags[XF_WORDS * l + XF_OVERFLOW];
        atomicMax(xstatus, ov);
    }
}

// ---------------------------------------------------------------------------------------
// padding for an empty index, and the multi-shard merge
// ---------------------------------------------------------------------------------------
__global__ void fill_padding_kernel(float* scores, long long* rows, long long count) {
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < count;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        scores[i] = -FLT_MAX;
        rows[i] = -1;
    }
}

// One CTA per query: the n_lists*k shard-local winners are sorted in shared memory by
// (score desc, global row asc) and the first k written out.  smem: P u64 keys.
__global__ void __launch_bounds__(SEL_THREADS)
merge_topk_kernel(long long nq, int k, int n_lists, const float* __restrict__ scores,
                  const long long* __restrict__ rows, long long scores_list_stride,
                  long long rows_list_stride, float* __restrict__ out_scores,
                  long long* __restrict__ out_rows, int P, const unsigned int* wait_flags,
                  unsigned int seq, long long* __restrict__ xstatus, long long q_first,
                  long long timeout_ns, const DynArgs* __restrict__ dyn) {
    if (dyn) {
        seq = dyn->seq;
        out_scores = dyn->ex_out_s;
        out_rows = dyn->ex_out_r;
    }
    extern __shared__ __align__(16) uint8_t msm[];
    unsigned long long* sbuf = reinterpret_cast<unsigned long long*>(msm);
    // owner mode: this rank merges queries [q_first, q_first + gridDim.x) of the search and
    // stores them compactly (row 0 of the output = query q_first)
    const long long q = q_first + blockIdx.x;
    const long long qo = blockIdx.x;
    const int total = n_lists * k;
    if (wait_flags) {
        // peer-direct exchange: list l was stored into this GPU's memory by rank l's finalize
        // kernel; rank l then published XF_RESULT = seq (release, system scope) and its overflow
        // count.  Wait for all of them, then merge as usual.
        wait_peer_flags(wait_flags, n_lists, XF_RESULT, seq, timeout_ns, xstatus);
        if (xstatus && blockIdx.x == 0 && threadIdx.x == 0) {
            long long ov = 0;
            for (int l = 0; l < n_lists; l++) ov += wait_flags[XF_WORDS * l + XF_OVERFLOW];
            atomicMax(xstatus, ov);
        }
    }
    for (int i = threadIdx.x; i < P; i += blockDim.x) {
        unsigned long long key = 0ull;
        if (i < total) {
            const int l = i / k, j = i - l * k;
            const long long src = q * k + j;
            const long long r = rows[l * rows_list_stride + src];
            if (r >= 0) key = make_key(scores[l * scores_list_stride + src], static_cast<uint32_t>(r));
        }
        sbuf[i] = key;
    }
    __syncthreads();
    block_bitonic_desc(sbuf, P);
    for (int j = threadIdx.x; j < k; j += blockDim.x) {
        const unsigned long long key = sbuf[j];
        float s = -FLT_MAX;
        long long r = -1;
        if ((key >> 32) != 0ull) { s = key_score(key); r = key_row(key); }
        out_scores[qo * k + j] = s;
        out_rows[qo * k + j] = r;
    }
}

}  // namespace b2ip
