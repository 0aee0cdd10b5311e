// coarse_kernel.cuh -- the scoring kernel of the tensor path.
//
// S = Q . X^T on the 5th-gen tensor cores (tcgen05.mma kind::f16, bf16 operands, fp32
// accumulate in TMEM) with the accumulator tile consumed in place by a per-query threshold
// filter: the score matrix never reaches HBM, only (score,row) pairs that beat the query's
// current threshold are appended to that query's candidate list.
//
// Replaces the sgemm + result-handler pair inside faiss::IndexFlatIP::search that the
// reference calls at src/index.py:42 (SURVEY.md 3.2: exhaustive_inner_product_blas).
//
// CTA = 256 threads, one CTA per SM (persistent over a static tile schedule):
//   warp 0 / lane 0 : TMA producer   (Q tile 128x64 + X tile 256x64 bf16 per k-block)
//   warp 1 / lane 0 : MMA issuer     (4 x tcgen05.mma 128x256x16 per k-block)
//   warp 2          : TMEM allocator (512 columns = 2 accumulator stages of 128x256 fp32)
//   warps 4..7      : filter epilogue (thread = query row; tcgen05.ld 32 columns at a time)
// Pipelines: STAGES-deep smem ring (full/empty mbarriers) between TMA and MMA, and a
// 2-deep TMEM ring (tmem_full/tmem_empty) between MMA and the epilogue, so the filter of
// tile i overlaps the MMAs of tile i+1.
#pragma once
#include "ptx_sm100.cuh"
#include "keys.cuh"

namespace b2ip {

constexpr int TILE_Q = 128;          // UMMA M  (queries per tile)
constexpr int TILE_X = 256;          // UMMA N  (corpus rows per tile)
constexpr int KBLOCK_BYTES = 128;    // one SWIZZLE_128B row: 64 bf16
constexpr int KBLOCK_ELEMS = 64;
constexpr int UMMA_K_BYTES = 32;     // 16 bf16 per tcgen05.mma
constexpr int STAGES = 4;
constexpr int A_STAGE_BYTES = TILE_Q * KBLOCK_BYTES;   // 16 KiB
constexpr int B_STAGE_BYTES = TILE_X * KBLOCK_BYTES;   // 32 KiB
constexpr int STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;
constexpr int COARSE_THREADS = 256;
constexpr int HIT_SLOTS = 8;         // per-thread staging slots for filter hits (shared memory)
constexpr int HIT_STAGE_BYTES = HIT_SLOTS * 128 * 8;
constexpr int COARSE_SMEM_BYTES =
    STAGES * STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/ + HIT_STAGE_BYTES;
constexpr uint32_t TMEM_COLS = 512;
// tcgen05 instruction descriptors, indexed by the operand format (SH_BF16 = 0, SH_F16 = 1)
constexpr uint32_t IDESC_SINGLE[2] = {ptx::umma_idesc(/*bf16*/ 1, TILE_Q, TILE_X),
                                      ptx::umma_idesc(/*f16*/ 0, TILE_Q, TILE_X)};
constexpr uint32_t IDESC_PAIR[2] = {ptx::umma_idesc(/*bf16*/ 1, 256, TILE_X),
                                    ptx::umma_idesc(/*f16*/ 0, 256, TILE_X)};

struct CoarseParams {
    int num_k_blocks;        // d_pad / 64
    int q_tiles;             // ceil(nq / 128)
    int x_tiles;             // tiles of 256 rows in this launch
    int gx;                  // x tiles per raster group (L2 reuse)
    int nq;
    long long x_row0;        // first corpus row of the launch (local row id)
    long long x_row_end;     // one past the last row that may be reported
    const float* thr;        // [nq] current per-query admission threshold (strict >)
    unsigned long long* cand;  // [nq, cap] candidate keys
    int* cnt;                // [nq] fill counters (may run past cap: overflow marker)
    int cap;
    float* dump;             // debug: [nq, dump_ld] raw scores, or nullptr
    long long dump_ld;
    unsigned long long hint_q, hint_x;   // L2 eviction-priority policies of the two TMA streams
    int dense;               // first slab of a search (every threshold is -inf): each column IS a
                             // hit, stored at list position = row - x_row0 without counters
                             // (the fill counters are preset to the slab size)
    uint32_t idesc;          // tcgen05 instruction descriptor (IDESC_SINGLE / IDESC_PAIR [format])
    int dbg;                 // perf experiments only (results are wrong when set):
                             // 1 = every tile loads corpus tile 0, 2 = no TMA loads, 4 = no filter
    uint32_t* gmax;          // coarse_stream_kernel<NQ, true> only: [nq, gridDim.x * 128] group maxima
    long long gstride;       // ... and the distance in rows between the sampled tiles (>= 128)
};

__device__ __forceinline__ void tile_coords(const CoarseParams& p, int t, int& qt, int& xt) {
    const int per_group = p.gx * p.q_tiles;
    const int xg = t / per_group;
    const int r = t - xg * per_group;
    const int rem = p.x_tiles - xg * p.gx;
    const int gx_eff = rem < p.gx ? rem : p.gx;
    qt = r / gx_eff;
    xt = xg * p.gx + (r - qt * gx_eff);
}

// v[j] for a run-time j without spilling v to local memory: 5-level tree of selects.
__device__ __forceinline__ uint32_t select32(const uint32_t (&v)[32], int j) {
    uint32_t a[16], b[8], c[4], d[2];
#pragma unroll
    for (int i = 0; i < 16; i++) a[i] = (j & 1) ? v[2 * i + 1] : v[2 * i];
#pragma unroll
    for (int i = 0; i < 8; i++) b[i] = (j & 2) ? a[2 * i + 1] : a[2 * i];
#pragma unroll
    for (int i = 0; i < 4; i++) c[i] = (j & 4) ? b[2 * i + 1] : b[2 * i];
#pragma unroll
    for (int i = 0; i < 2; i++) d[i] = (j & 8) ? c[2 * i + 1] : c[2 * i];
    return (j & 16) ? d[1] : d[0];
}

// Appends a thread's staged hits to its query's candidate list: ONE counter bump per flush.
__device__ __forceinline__ void flush_hits(const CoarseParams& p, int q,
                                           const unsigned long long* my_stage, int n) {
    const int slot = atomicAdd(p.cnt + q, n);
    unsigned long long* dst = p.cand + static_cast<long long>(q) * p.cap;
    for (int i = 0; i < n; i++)
        if (slot + i < p.cap) dst[slot + i] = my_stage[i * 128];
}

// The fused filter: one thread = one query row (TMEM lane) of a 128 x 256 fp32 accumulator.
// 32 columns at a time: tcgen05.ld, FMNMX3 tree -> chunk maximum, one compare against the
// row's threshold.  Only if it passes (rare): branch-free hit mask, hits staged in shared
// memory (flushed once per tile, after the accumulator is released) -- or, for dense chunks
// (early slabs), appended straight from registers with one counter bump per chunk.
// kFilter (filtered search): a hit is admitted only when its row's bit is set in `allow`.  Slabs
// start at multiples of TILE_X (tensor_search), so the 32 rows of a chunk are exactly one word.
template <bool kFilter = false>
__device__ __forceinline__ void filter_accumulator(const CoarseParams& p, int q, float thr,
                                                   uint32_t taddr, long long x_row, int n_valid,
                                                   unsigned long long* my_stage, int& n_staged,
                                                   const uint32_t* allow = nullptr) {
#pragma unroll 1
    for (int c = 0; c < TILE_X / 32; c++) {
        uint32_t v[32];
        ptx::tmem_ld_32x32(taddr + c * 32, v);
        ptx::tmem_ld_wait();
        float m = __uint_as_float(v[0]);
#pragma unroll
        for (int j = 1; j < 32; j++) m = fmaxf(m, __uint_as_float(v[j]));
        if (m > thr) {
            uint32_t mask = 0;
#pragma unroll
            for (int j = 0; j < 32; j++) mask |= (__uint_as_float(v[j]) > thr) ? (1u << j) : 0u;
            const int vcols = n_valid - c * 32;          // columns of this chunk in range
            if (vcols < 32) mask &= vcols > 0 ? ((1u << vcols) - 1u) : 0u;
            const uint32_t row0 = static_cast<uint32_t>(x_row) + c * 32;
            if constexpr (kFilter) {
                if (mask) mask &= row_word(allow, row0);   // a set bit means row0 < x_row_end
            }
            const int nh = __popc(mask);
            if (n_staged + nh > HIT_SLOTS) {
                int slot = atomicAdd(p.cnt + q, nh);
                unsigned long long* dst = p.cand + static_cast<long long>(q) * p.cap;
                while (mask) {
                    const int j = __ffs(mask) - 1;
                    mask &= mask - 1;
                    const uint32_t bits = select32(v, j);
                    if (slot < p.cap) dst[slot] = make_key(__uint_as_float(bits), row0 + j);
                    slot++;
                }
            } else {
                while (mask) {
                    const int j = __ffs(mask) - 1;
                    mask &= mask - 1;
                    const uint32_t bits = select32(v, j);
                    my_stage[n_staged * 128] = make_key(__uint_as_float(bits), row0 + j);
                    n_staged++;
                }
            }
        }
    }
}

// First slab: no threshold exists yet, so every in-range column is a candidate.  Its list
// position is its row offset inside the slab: no atomics, no hit extraction, 16-byte stores.
__device__ __forceinline__ void dense_store_accumulator(const CoarseParams& p, int q, uint32_t taddr,
                                                        long long x_row, int n_valid) {
    unsigned long long* dst =
        p.cand + static_cast<long long>(q < p.nq ? q : 0) * p.cap + (x_row - p.x_row0);
#pragma unroll 1
    for (int c = 0; c < TILE_X / 32; c++) {
        uint32_t v[32];
        ptx::tmem_ld_32x32(taddr + c * 32, v);
        ptx::tmem_ld_wait();
        if (q < p.nq) {
            const uint32_t row0 = static_cast<uint32_t>(x_row) + c * 32;
            if (n_valid - c * 32 >= 32) {
#pragma unroll
                for (int j = 0; j < 32; j += 2) {
                    ulonglong2 two;
                    two.x = make_key(__uint_as_float(v[j]), row0 + j);
                    two.y = make_key(__uint_as_float(v[j + 1]), row0 + j + 1);
                    *reinterpret_cast<ulonglong2*>(dst + c * 32 + j) = two;
                }
            } else {
#pragma unroll
                for (int j = 0; j < 32; j++)
                    if (c * 32 + j < n_valid) dst[c * 32 + j] = make_key(__uint_as_float(v[j]), row0 + j);
            }
        }
    }
}

// The scoring kernels below are bodies shared by two entry points each: the search kernel and,
// with kFilter, its filtered twin (`..._bitmap`), which takes the allowed-row bitmap as one more
// kernel argument.  (A CoarseParams field would grow the struct and move the `stages` argument
// of coarse_stream_kernel: the unfiltered kernels would no longer compile to the same code.)
template <bool kDump, bool kFilter>
__device__ __forceinline__ void coarse_filter_body(const CUtensorMap& tmap_q, const CUtensorMap& tmap_x,
                                                   const CoarseParams p, const uint32_t* allow) {
    extern __shared__ uint8_t smem_raw[];
    // SWIZZLE_128B operand tiles need 1024-byte alignment.
    uint8_t* smem = reinterpret_cast<uint8_t*>(
        (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
    uint8_t* smem_a = smem;
    uint8_t* smem_b = smem + STAGES * A_STAGE_BYTES;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);
    uint64_t* full_bar = bars;                 // [STAGES]
    uint64_t* empty_bar = bars + STAGES;       // [STAGES]
    uint64_t* tfull_bar = bars + 2 * STAGES;   // [2]
    uint64_t* tempty_bar = bars + 2 * STAGES + 2;  // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);
    // hit staging: slot i of epilogue thread e lives at hit_stage[i * 128 + e] (conflict-free)
    unsigned long long* hit_stage =
        reinterpret_cast<unsigned long long*>(smem + STAGES * STAGE_BYTES + 256);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int total_tiles = p.q_tiles * p.x_tiles;

    if (warp == 0 && lane == 0) {
        ptx::prefetch_tmap(&tmap_q);
        ptx::prefetch_tmap(&tmap_x);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < STAGES; s++) {
            ptx::mbar_init(&full_bar[s], 1);
            ptx::mbar_init(&empty_bar[s], 1);
        }
        for (int s = 0; s < 2; s++) {
            ptx::mbar_init(&tfull_bar[s], 1);
            ptx::mbar_init(&tempty_bar[s], 128);
        }
        ptx::fence_mbar_init();
    }
    if (warp == 2) ptx::tmem_alloc<TMEM_COLS>(tmem_slot);
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            // ===================== TMA producer =====================
            int stage = 0;
            uint32_t phase = 0;
            for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
                int qt, xt;
                tile_coords(p, t, qt, xt);
                const int q_row = qt * TILE_Q;
                const long long x_row =
                    (p.dbg & 1) ? 0 : p.x_row0 + static_cast<long long>(xt) * TILE_X;
                for (int kb = 0; kb < p.num_k_blocks; kb++) {
                    ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
                    if (p.dbg & 2) {
                        ptx::mbar_arrive(&full_bar[stage]);
                        if (++stage == STAGES) { stage = 0; phase ^= 1; }
                        continue;
                    }
                    ptx::mbar_expect_tx(&full_bar[stage], STAGE_BYTES);
                    ptx::tma_load_2d(smem_a + stage * A_STAGE_BYTES, &tmap_q, &full_bar[stage],
                                     kb * KBLOCK_ELEMS, q_row, p.hint_q);
                    ptx::tma_load_2d(smem_b + stage * B_STAGE_BYTES, &tmap_x, &full_bar[stage],
                                     kb * KBLOCK_ELEMS, static_cast<int32_t>(x_row), p.hint_x);
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            // ===================== MMA issuer =====================
            int stage = 0;
            uint32_t phase = 0;
            int as = 0;
            uint32_t aphase = 0;
            for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
                ptx::mbar_wait(&tempty_bar[as], aphase ^ 1);
                ptx::tc_fence_after();
                const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(as * TILE_X);
                for (int kb = 0; kb < p.num_k_blocks; kb++) {
                    ptx::mbar_wait(&full_bar[stage], phase);
                    ptx::tc_fence_after();
                    const uint32_t a_addr = ptx::smem_u32(smem_a + stage * A_STAGE_BYTES);
                    const uint32_t b_addr = ptx::smem_u32(smem_b + stage * B_STAGE_BYTES);
#pragma unroll
                    for (int k = 0; k < KBLOCK_BYTES / UMMA_K_BYTES; k++) {
                        const uint64_t adesc = ptx::umma_desc_k_sw128(a_addr + k * UMMA_K_BYTES);
                        const uint64_t bdesc = ptx::umma_desc_k_sw128(b_addr + k * UMMA_K_BYTES);
                        ptx::mma_f16_ss(d_tmem, adesc, bdesc, p.idesc, (kb | k) != 0);
                    }
                    ptx::tc_commit(&empty_bar[stage]);   // smem slot reusable once MMAs retire
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
                ptx::tc_commit(&tfull_bar[as]);          // accumulator complete
                if (++as == 2) { as = 0; aphase ^= 1; }
            }
        }
    } else if (warp >= 4) {
        // ===================== filter epilogue =====================
        const int wq = warp & 3;                         // TMEM lane quarter of this warp
        int as = 0;
        uint32_t aphase = 0;
        for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
            int qt, xt;
            tile_coords(p, t, qt, xt);
            const int q = qt * TILE_Q + wq * 32 + lane;
            unsigned long long* my_stage = hit_stage + (wq * 32 + lane);
            int n_staged = 0;
            const long long x_row = p.x_row0 + static_cast<long long>(xt) * TILE_X;
            const long long left = p.x_row_end - x_row;
            const int n_valid = left < TILE_X ? static_cast<int>(left) : TILE_X;
            float thr = __int_as_float(0x7f800000);      // +inf: padding rows never report
            if (q < p.nq) thr = kDump ? 0.f : __ldg(p.thr + q);

            ptx::mbar_wait(&tfull_bar[as], aphase);
            ptx::tc_fence_after();
            const uint32_t taddr =
                tmem_base + (static_cast<uint32_t>(wq * 32) << 16) + static_cast<uint32_t>(as * TILE_X);
            if (kDump) {
#pragma unroll 1
                for (int c = 0; c < TILE_X / 32; c++) {
                    uint32_t v[32];
                    ptx::tmem_ld_32x32(taddr + c * 32, v);
                    ptx::tmem_ld_wait();
                    if (q < p.nq) {
#pragma unroll
                        for (int j = 0; j < 32; j++) {
                            const int col = c * 32 + j;
                            if (col < n_valid)
                                p.dump[static_cast<long long>(q) * p.dump_ld +
                                       static_cast<long long>(xt) * TILE_X + col] = __uint_as_float(v[j]);
                        }
                    }
                }
            } else if (p.dense) {
                dense_store_accumulator(p, q, taddr, x_row, n_valid);
            } else if (!(p.dbg & 4)) {
                filter_accumulator<kFilter>(p, q, thr, taddr, x_row, n_valid, my_stage, n_staged, allow);
            }
            // hand the accumulator back before touching global memory: the (latency-bound)
            // counter bump + key stores then overlap the MMAs of the following tiles
            ptx::tc_fence_before();
            ptx::mbar_arrive(&tempty_bar[as]);
            if (++as == 2) { as = 0; aphase ^= 1; }
            if (!kDump && n_staged) flush_hits(p, q, my_stage, n_staged);
        }
    }

    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        ptx::tc_fence_after();
        ptx::tmem_dealloc<TMEM_COLS>(tmem_base);
    }
}

template <bool kDump>
__global__ void __launch_bounds__(COARSE_THREADS, 1)
coarse_filter_kernel(const __grid_constant__ CUtensorMap tmap_q,
                     const __grid_constant__ CUtensorMap tmap_x, const CoarseParams p) {
    coarse_filter_body<kDump, false>(tmap_q, tmap_x, p, nullptr);
}

__global__ void __launch_bounds__(COARSE_THREADS, 1)
coarse_filter_kernel_bitmap(const __grid_constant__ CUtensorMap tmap_q,
                            const __grid_constant__ CUtensorMap tmap_x, const CoarseParams p,
                            const uint32_t* __restrict__ allow) {
    coarse_filter_body<false, true>(tmap_q, tmap_x, p, allow);
}

// =======================================================================================
// CTA-pair variant (cta_group::2): one 256-query x 256-row tile per cluster of two SMs.
// Each CTA stages ITS 128 query rows (A half) and ITS 128 corpus rows (B half) -- 32 KiB per
// k-block instead of 48 KiB, a third less L2->SM and smem->tensor-core operand traffic per
// flop -- the leader CTA issues tcgen05.mma.cta_group::2 (M = 256), each CTA filters the 128
// accumulator rows that land in its own TMEM.
//   full[s]   : leader's barrier; leader arrives with expect_tx(64 KiB), both CTAs' TMA loads
//               complete_tx on it
//   empty[s]  : per CTA; tcgen05.commit multicast to both when the stage's MMAs retire
//   tfull[a]  : per CTA; commit multicast when an accumulator is complete
//   tempty[a] : leader's barrier; 256 arrivals = epilogue threads of both CTAs
// =======================================================================================
constexpr int PAIR_STAGES = 6;
constexpr int PAIR_HALF_BYTES = 128 * KBLOCK_BYTES;            // 16 KiB: 128 rows x 128 B
constexpr int PAIR_STAGE_BYTES = 2 * PAIR_HALF_BYTES;          // A half + B half per CTA
constexpr int PAIR_SMEM_BYTES =
    PAIR_STAGES * PAIR_STAGE_BYTES + 1024 + 256 + HIT_STAGE_BYTES;

template <bool kFilter>
__device__ __forceinline__ void coarse_filter_pair_body(const CUtensorMap& tmap_q, const CUtensorMap& tmap_x,
                                                        const CoarseParams p, const uint32_t* allow) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>(
        (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
    uint8_t* smem_a = smem;
    uint8_t* smem_b = smem + PAIR_STAGES * PAIR_HALF_BYTES;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + PAIR_STAGES * PAIR_STAGE_BYTES);
    uint64_t* full_bar = bars;                            // [PAIR_STAGES]
    uint64_t* empty_bar = bars + PAIR_STAGES;             // [PAIR_STAGES]
    uint64_t* tfull_bar = bars + 2 * PAIR_STAGES;         // [2]
    uint64_t* tempty_bar = bars + 2 * PAIR_STAGES + 2;    // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * PAIR_STAGES + 4);
    unsigned long long* hit_stage =
        reinterpret_cast<unsigned long long*>(smem + PAIR_STAGES * PAIR_STAGE_BYTES + 256);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint32_t rank = ptx::cluster_ctarank();         // 0 = leader
    const int cluster_id = blockIdx.x >> 1;
    const int n_clusters = gridDim.x >> 1;
    // p.q_tiles counts 256-query pair tiles here
    const int total_tiles = p.q_tiles * p.x_tiles;

    if (warp == 0 && lane == 0) {
        ptx::prefetch_tmap(&tmap_q);
        ptx::prefetch_tmap(&tmap_x);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < PAIR_STAGES; s++) {
            ptx::mbar_init(&full_bar[s], 1);
            ptx::mbar_init(&empty_bar[s], 1);
        }
        for (int s = 0; s < 2; s++) {
            ptx::mbar_init(&tfull_bar[s], 1);
            ptx::mbar_init(&tempty_bar[s], 256);
        }
        ptx::fence_mbar_init();
    }
    if (warp == 2) ptx::tmem_alloc_pair<TMEM_COLS>(tmem_slot);
    ptx::tc_fence_before();
    __syncthreads();
    ptx::cluster_sync_all();              // peer barriers initialised before any remote signal
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            // ===================== TMA producer (both CTAs) =====================
            int stage = 0;
            uint32_t phase = 0;
            for (int t = cluster_id; t < total_tiles; t += n_clusters) {
                int qt, xt;
                tile_coords(p, t, qt, xt);
                const int q_row = qt * 256 + static_cast<int>(rank) * 128;
                const long long x_row =
                    p.x_row0 + static_cast<long long>(xt) * TILE_X + static_cast<long long>(rank) * 128;
                for (int kb = 0; kb < p.num_k_blocks; kb++) {
                    ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
                    if (rank == 0) ptx::mbar_expect_tx(&full_bar[stage], 2 * PAIR_STAGE_BYTES);
                    ptx::tma_load_2d_pair(smem_a + stage * PAIR_HALF_BYTES, &tmap_q, &full_bar[stage],
                                          kb * KBLOCK_ELEMS, q_row, p.hint_q);
                    ptx::tma_load_2d_pair(smem_b + stage * PAIR_HALF_BYTES, &tmap_x, &full_bar[stage],
                                          kb * KBLOCK_ELEMS, static_cast<int32_t>(x_row), p.hint_x);
                    if (++stage == PAIR_STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0 && rank == 0) {
            // ===================== MMA issuer (leader CTA only) =====================
            int stage = 0;
            uint32_t phase = 0;
            int as = 0;
            uint32_t aphase = 0;
            for (int t = cluster_id; t < total_tiles; t += n_clusters) {
                ptx::mbar_wait(&tempty_bar[as], aphase ^ 1);
                ptx::tc_fence_after();
                const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(as * TILE_X);
                for (int kb = 0; kb < p.num_k_blocks; kb++) {
                    ptx::mbar_wait(&full_bar[stage], phase);
                    ptx::tc_fence_after();
                    const uint32_t a_addr = ptx::smem_u32(smem_a + stage * PAIR_HALF_BYTES);
                    const uint32_t b_addr = ptx::smem_u32(smem_b + stage * PAIR_HALF_BYTES);
#pragma unroll
                    for (int k = 0; k < KBLOCK_BYTES / UMMA_K_BYTES; k++) {
                        const uint64_t adesc = ptx::umma_desc_k_sw128(a_addr + k * UMMA_K_BYTES);
                        const uint64_t bdesc = ptx::umma_desc_k_sw128(b_addr + k * UMMA_K_BYTES);
                        ptx::mma_f16_ss_pair(d_tmem, adesc, bdesc, p.idesc, (kb | k) != 0);
                    }
                    ptx::tc_commit_pair(&empty_bar[stage], 0x3);
                    if (++stage == PAIR_STAGES) { stage = 0; phase ^= 1; }
                }
                ptx::tc_commit_pair(&tfull_bar[as], 0x3);
                if (++as == 2) { as = 0; aphase ^= 1; }
            }
        }
    } else if (warp >= 4) {
        // ===================== filter epilogue (both CTAs, own 128 rows) =====================
        const int wq = warp & 3;
        int as = 0;
        uint32_t aphase = 0;
        const uint32_t tempty_leader0 = ptx::mapa_u32(&tempty_bar[0], 0);
        const uint32_t tempty_leader1 = ptx::mapa_u32(&tempty_bar[1], 0);
        for (int t = cluster_id; t < total_tiles; t += n_clusters) {
            int qt, xt;
            tile_coords(p, t, qt, xt);
            const int q = qt * 256 + static_cast<int>(rank) * 128 + wq * 32 + lane;
            unsigned long long* my_stage = hit_stage + (wq * 32 + lane);
            int n_staged = 0;
            const long long x_row = p.x_row0 + static_cast<long long>(xt) * TILE_X;
            const long long left = p.x_row_end - x_row;
            const int n_valid = left < TILE_X ? static_cast<int>(left) : TILE_X;
            float thr = __int_as_float(0x7f800000);
            if (q < p.nq) thr = __ldg(p.thr + q);

            ptx::mbar_wait(&tfull_bar[as], aphase);
            ptx::tc_fence_after();
            const uint32_t taddr =
                tmem_base + (static_cast<uint32_t>(wq * 32) << 16) + static_cast<uint32_t>(as * TILE_X);
            if (p.dense) dense_store_accumulator(p, q, taddr, x_row, n_valid);
            else if (!(p.dbg & 4))
                filter_accumulator<kFilter>(p, q, thr, taddr, x_row, n_valid, my_stage, n_staged, allow);
            ptx::tc_fence_before();
            ptx::mbar_arrive_cluster(as == 0 ? tempty_leader0 : tempty_leader1);
            if (++as == 2) { as = 0; aphase ^= 1; }
            if (n_staged) flush_hits(p, q, my_stage, n_staged);
        }
    }

    // nobody may leave (or free TMEM) while the peer can still signal / be read
    ptx::tc_fence_before();
    __syncthreads();
    ptx::cluster_sync_all();
    if (warp == 2) {
        ptx::tc_fence_after();
        ptx::tmem_dealloc_pair<TMEM_COLS>(tmem_base);
    }
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(COARSE_THREADS, 1)
coarse_filter_pair_kernel(const __grid_constant__ CUtensorMap tmap_q,
                          const __grid_constant__ CUtensorMap tmap_x, const CoarseParams p) {
    coarse_filter_pair_body<false>(tmap_q, tmap_x, p, nullptr);
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(COARSE_THREADS, 1)
coarse_filter_pair_kernel_bitmap(const __grid_constant__ CUtensorMap tmap_q,
                                 const __grid_constant__ CUtensorMap tmap_x, const CoarseParams p,
                                 const uint32_t* __restrict__ allow) {
    coarse_filter_pair_body<true>(tmap_q, tmap_x, p, allow);
}

// =======================================================================================
// Streaming variant for small query batches (nq <= 64): BASELINE config 5, the HBM-bound
// latency regime.  Operands are swapped with respect to the kernels above: the CORPUS tile is
// the M side of the MMA (128 rows = 128 TMEM lanes) and the padded query batch the N side
// (NQ = 32 or 64 columns), so a tile costs 128 x NQ x d MACs instead of 128 x 256 x d for 256
// rows -- 2-4x less tensor-core work (and power: this regime is power-capped too) for the same
// bytes.  The whole query batch stays RESIDENT in shared memory (loaded once per CTA), so the
// only L2->SM stream is the corpus itself: STAGES x 16 KiB of TMA loads in flight per SM.
//   warp 0 / lane 0 : TMA producer (queries once, then 128-row corpus tiles, k-block by k-block)
//   warp 1 / lane 0 : MMA issuer   (4 x tcgen05.mma 128 x NQ x 16 per k-block)
//   warp 2          : TMEM allocator (4 accumulator stages of NQ columns)
//   warps 4..7      : filter epilogue; thread = corpus row, its NQ scores against the NQ
//                     per-query thresholds held in registers
// =======================================================================================
constexpr int STREAM_TILE_X = 128;
constexpr int STREAM_MAX_STAGES = 12;   // corpus stages the barrier area holds
constexpr int STREAM_STAGES = 8;        // stages run when they fit (5 - 12 measure the same: DESIGN 4.1d)
constexpr int STREAM_ACC = 4;
constexpr int STREAM_X_STAGE_BYTES = STREAM_TILE_X * KBLOCK_BYTES;   // 16 KiB
constexpr int STREAM_MISC_BYTES = 1024 /*align*/ + 320 /*barriers*/;

// kGroupMax = the threshold bootstrap of a small batch: one launch over a SAMPLE of x_tiles tiles of
// 128 rows (x_tiles >= the grid: every CTA sees a tile) spread evenly over the corpus, tile t = rows
// [t * gstride, +128).  Nothing is filtered or listed; epilogue thread (CTA b, row slot s) keeps,
// per query, the maximum ordered score over the rows it sees -- row s of tiles b, b + grid, ... ,
// i.e. a GROUP of rows far apart (neighbouring rows, which score alike in a real corpus, fall
// into different groups) -- and stores it to gmax[q][b*128 + s].  The groups are
// disjoint, so the k-th largest group maximum is a lower bound of the k-th best score of the corpus:
// bootstrap_threshold_kernel turns it into the admission threshold of the ONE filtered slab that
// follows (instead of dense slab -> refresh -> small slab -> refresh -> main slab).
template <int NQ, bool kGroupMax, bool kFilter>
__device__ __forceinline__ void coarse_stream_body(const CUtensorMap& tmap_q, const CUtensorMap& tmap_x,
                                                   const CoarseParams p, const int stages,
                                                   const uint32_t* allow) {
    static_assert(NQ == 32 || NQ == 64, "query batch is padded to 32 or 64 columns");
    static_assert(!(kGroupMax && kFilter), "a filtered search takes no threshold bootstrap");
    constexpr uint32_t kTmemCols = STREAM_ACC * NQ;                  // 128 or 256: powers of two
    constexpr int Q_KB_BYTES = NQ * KBLOCK_BYTES;                     // one k-block of the batch
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>(
        (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
    uint8_t* smem_x = smem;                                           // [stages][128 x 128 B]
    uint8_t* smem_q = smem + stages * STREAM_X_STAGE_BYTES;           // [num_k_blocks][NQ x 128 B]
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_q + p.num_k_blocks * Q_KB_BYTES);
    uint64_t* full_bar = bars;                                        // [STREAM_MAX_STAGES]
    uint64_t* empty_bar = bars + STREAM_MAX_STAGES;                   // [STREAM_MAX_STAGES]
    uint64_t* tfull_bar = bars + 2 * STREAM_MAX_STAGES;               // [STREAM_ACC]
    uint64_t* tempty_bar = bars + 2 * STREAM_MAX_STAGES + STREAM_ACC; // [STREAM_ACC]
    uint64_t* qfull_bar = bars + 2 * STREAM_MAX_STAGES + 2 * STREAM_ACC;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(qfull_bar + 1);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int total_tiles = p.x_tiles;                                // tiles of 128 corpus rows

    if (warp == 0 && lane == 0) {
        ptx::prefetch_tmap(&tmap_q);
        ptx::prefetch_tmap(&tmap_x);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < STREAM_MAX_STAGES; s++) {
            ptx::mbar_init(&full_bar[s], 1);
            ptx::mbar_init(&empty_bar[s], 1);
        }
        for (int s = 0; s < STREAM_ACC; s++) {
            ptx::mbar_init(&tfull_bar[s], 1);
            ptx::mbar_init(&tempty_bar[s], 128);
        }
        ptx::mbar_init(qfull_bar, 1);
        ptx::fence_mbar_init();
    }
    if (warp == 2) ptx::tmem_alloc<kTmemCols>(tmem_slot);
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            // ===================== TMA producer =====================
            ptx::mbar_expect_tx(qfull_bar, static_cast<uint32_t>(p.num_k_blocks * Q_KB_BYTES));
            for (int kb = 0; kb < p.num_k_blocks; kb++)
                ptx::tma_load_2d(smem_q + kb * Q_KB_BYTES, &tmap_q, qfull_bar, kb * KBLOCK_ELEMS, 0,
                                 p.hint_q);
            int stage = 0;
            uint32_t phase = 0;
            for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
                const long long x_row = p.x_row0 + static_cast<long long>(t) * (kGroupMax ? p.gstride : STREAM_TILE_X);
                for (int kb = 0; kb < p.num_k_blocks; kb++) {
                    ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
                    ptx::mbar_expect_tx(&full_bar[stage], STREAM_X_STAGE_BYTES);
                    ptx::tma_load_2d(smem_x + stage * STREAM_X_STAGE_BYTES, &tmap_x, &full_bar[stage],
                                     kb * KBLOCK_ELEMS, static_cast<int32_t>(x_row), p.hint_x);
                    if (++stage == stages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            // ===================== MMA issuer =====================
            ptx::mbar_wait(qfull_bar, 0);
            ptx::tc_fence_after();
            int stage = 0;
            uint32_t phase = 0;
            int as = 0;
            uint32_t aphase = 0;
            for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
                ptx::mbar_wait(&tempty_bar[as], aphase ^ 1);
                ptx::tc_fence_after();
                const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(as * NQ);
                for (int kb = 0; kb < p.num_k_blocks; kb++) {
                    ptx::mbar_wait(&full_bar[stage], phase);
                    ptx::tc_fence_after();
                    const uint32_t a_addr = ptx::smem_u32(smem_x + stage * STREAM_X_STAGE_BYTES);
                    const uint32_t b_addr = ptx::smem_u32(smem_q + kb * Q_KB_BYTES);
#pragma unroll
                    for (int k = 0; k < KBLOCK_BYTES / UMMA_K_BYTES; k++) {
                        const uint64_t adesc = ptx::umma_desc_k_sw128(a_addr + k * UMMA_K_BYTES);
                        const uint64_t bdesc = ptx::umma_desc_k_sw128(b_addr + k * UMMA_K_BYTES);
                        ptx::mma_f16_ss(d_tmem, adesc, bdesc, p.idesc, (kb | k) != 0);
                    }
                    ptx::tc_commit(&empty_bar[stage]);
                    if (++stage == stages) { stage = 0; phase ^= 1; }
                }
                ptx::tc_commit(&tfull_bar[as]);
                if (++as == STREAM_ACC) { as = 0; aphase ^= 1; }
            }
        }
    } else if (warp >= 4) {
        // ===================== filter epilogue: thread = corpus row =====================
        const int wq = warp & 3;
        int as = 0;
        uint32_t aphase = 0;
        if constexpr (kGroupMax) {
            uint32_t gm[NQ];
#pragma unroll
            for (int j = 0; j < NQ; j++) gm[j] = 0u;                   // order(NaN): below every score
            for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
                const long long row = p.x_row0 + static_cast<long long>(t) * p.gstride + wq * 32 + lane;
                const bool row_ok = row < p.x_row_end;
                ptx::mbar_wait(&tfull_bar[as], aphase);
                ptx::tc_fence_after();
                const uint32_t taddr =
                    tmem_base + (static_cast<uint32_t>(wq * 32) << 16) + static_cast<uint32_t>(as * NQ);
#pragma unroll
                for (int c = 0; c < NQ / 32; c++) {
                    uint32_t v[32];
                    ptx::tmem_ld_32x32(taddr + c * 32, v);
                    ptx::tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 32; j++) {
                        const uint32_t o = row_ok ? order_f32(__uint_as_float(v[j])) : 0u;
                        gm[c * 32 + j] = max(gm[c * 32 + j], o);
                    }
                }
                ptx::tc_fence_before();
                ptx::mbar_arrive(&tempty_bar[as]);
                if (++as == STREAM_ACC) { as = 0; aphase ^= 1; }
            }
            // for a fixed query the 128 epilogue threads of a CTA store 128 consecutive words
            const long long groups = static_cast<long long>(gridDim.x) * STREAM_TILE_X;
            uint32_t* dst = p.gmax + static_cast<long long>(blockIdx.x) * STREAM_TILE_X + wq * 32 + lane;
#pragma unroll
            for (int j = 0; j < NQ; j++)
                if (j < p.nq) dst[static_cast<long long>(j) * groups] = gm[j];
        } else {
        float thr_r[NQ];
#pragma unroll
        for (int j = 0; j < NQ; j++)
            thr_r[j] = j < p.nq ? __ldg(p.thr + j) : __int_as_float(0x7f800000);   // +inf: padding
        for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
            const long long row = p.x_row0 + static_cast<long long>(t) * STREAM_TILE_X + wq * 32 + lane;
            bool row_ok = row < p.x_row_end;
            if constexpr (kFilter) row_ok = row_ok && row_allowed(allow, row);
            ptx::mbar_wait(&tfull_bar[as], aphase);
            ptx::tc_fence_after();
            const uint32_t taddr =
                tmem_base + (static_cast<uint32_t>(wq * 32) << 16) + static_cast<uint32_t>(as * NQ);
#pragma unroll
            for (int c = 0; c < NQ / 32; c++) {
                uint32_t v[32];
                ptx::tmem_ld_32x32(taddr + c * 32, v);
                ptx::tmem_ld_wait();
                if (p.dense) {
                    // first slab: list position = row offset in the slab; for a fixed query the 32
                    // lanes of a warp store 32 consecutive keys
                    if (row_ok) {
#pragma unroll
                        for (int j = 0; j < 32; j++)
                            if (c * 32 + j < p.nq)
                                p.cand[static_cast<long long>(c * 32 + j) * p.cap + (row - p.x_row0)] =
                                    make_key(__uint_as_float(v[j]), static_cast<uint32_t>(row));
                    }
                } else {
                    uint32_t mask = 0;
#pragma unroll
                    for (int j = 0; j < 32; j++)
                        mask |= (__uint_as_float(v[j]) > thr_r[c * 32 + j]) ? (1u << j) : 0u;
                    if (!row_ok) mask = 0;
                    while (mask) {
                        const int j = __ffs(mask) - 1;
                        mask &= mask - 1;
                        const int q = c * 32 + j;
                        const uint32_t bits = select32(v, j);
                        const int slot = atomicAdd(p.cnt + q, 1);
                        if (slot < p.cap)
                            p.cand[static_cast<long long>(q) * p.cap + slot] =
                                make_key(__uint_as_float(bits), static_cast<uint32_t>(row));
                    }
                }
            }
            ptx::tc_fence_before();
            ptx::mbar_arrive(&tempty_bar[as]);
            if (++as == STREAM_ACC) { as = 0; aphase ^= 1; }
        }
        }   // !kGroupMax
    }

    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        ptx::tc_fence_after();
        ptx::tmem_dealloc<kTmemCols>(tmem_base);
    }
}

template <int NQ, bool kGroupMax = false>
__global__ void __launch_bounds__(COARSE_THREADS, 1)
coarse_stream_kernel(const __grid_constant__ CUtensorMap tmap_q,
                     const __grid_constant__ CUtensorMap tmap_x, const CoarseParams p,
                     const int stages) {
    coarse_stream_body<NQ, kGroupMax, false>(tmap_q, tmap_x, p, stages, nullptr);
}

template <int NQ>
__global__ void __launch_bounds__(COARSE_THREADS, 1)
coarse_stream_kernel_bitmap(const __grid_constant__ CUtensorMap tmap_q,
                            const __grid_constant__ CUtensorMap tmap_x, const CoarseParams p,
                            const int stages, const uint32_t* __restrict__ allow) {
    coarse_stream_body<NQ, false, true>(tmap_q, tmap_x, p, stages, allow);
}

}  // namespace b2ip
