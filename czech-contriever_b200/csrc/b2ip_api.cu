// b2ip_api.cu -- host side of libb2ip.so: index state in HBM, slab scheduling of the
// tensor path, the exact fallback, and the C ABI declared in include/b2ip.h.
//
// HBM layout of one index (= one row shard on one GPU):
//   x32 [n, d]      fp32 master rows   (rescore, export, exact path)   -- what faiss keeps on host
//   x16 [n, d_pad]  bf16 shadow rows   (operand of the tcgen05 coarse GEMM), d_pad = ceil64(d)
//   norm_stats[2]   max ||x||^2, max ||x - bf16(x)||^2 (error bound of the coarse scores)
// Per search (grow-only workspace): bf16 queries, eps2/thr/cnt/kept/flags per query, candidate
// lists [nq_batch, cap] of 64-bit keys, device outputs.
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/b2ip.h"
#include "coarse_kernel.cuh"
#include "select_kernels.cuh"

using namespace b2ip;

// operand type of the coarse pass when the index keeps fp32 master rows (b2ip_set_option
// "shadow_f16" / env B2IP_SHADOW override it)
#ifndef B2IP_DEFAULT_SHADOW
#define B2IP_DEFAULT_SHADOW SH_BF16
#endif
static constexpr int SH_DEFAULT_F32_STORE = B2IP_DEFAULT_SHADOW;
static constexpr int MAX_SMEM_OPTIN = 227 * 1024;     // dynamic shared memory a CTA may opt in to (sm_100)

namespace {

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                    const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                    const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

thread_local std::string g_create_error;

struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
};

}  // namespace

namespace { class CopyPool; }

// Row storage that grows IN PLACE: a virtual address range sized for the whole device is reserved
// once and physical chunks are mapped behind the rows as they arrive (CUDA virtual memory
// management), so appending never needs old and new copy resident together -- a 97 GB fp32 index
// grows chunk by chunk to exactly its final size (cudaMalloc + copy would need 1.5-2x transiently
// and fail on the last steps).  Driver entry points are resolved at run time (no libcuda link).
struct VmmApi {
    CUresult (*getGranularity)(size_t*, const CUmemAllocationProp*, CUmemAllocationGranularity_flags) = nullptr;
    CUresult (*addressReserve)(CUdeviceptr*, size_t, size_t, CUdeviceptr, unsigned long long) = nullptr;
    CUresult (*create)(CUmemGenericAllocationHandle*, size_t, const CUmemAllocationProp*, unsigned long long) = nullptr;
    CUresult (*map)(CUdeviceptr, size_t, size_t, CUmemGenericAllocationHandle, unsigned long long) = nullptr;
    CUresult (*setAccess)(CUdeviceptr, size_t, const CUmemAccessDesc*, size_t) = nullptr;
    CUresult (*unmap)(CUdeviceptr, size_t) = nullptr;
    CUresult (*release)(CUmemGenericAllocationHandle) = nullptr;
    CUresult (*addressFree)(CUdeviceptr, size_t) = nullptr;
    bool ok = false;
};
struct VBuf {
    CUdeviceptr base = 0;
    size_t reserved = 0, mapped = 0;
    std::vector<std::pair<CUmemGenericAllocationHandle, size_t>> chunks;
};

struct b2ip_index_s {
    void* pin[2] = {nullptr, nullptr};    // pinned staging of host_to_device
    cudaEvent_t pin_ev[2] = {nullptr, nullptr};
    int pin_next = 0;
    CopyPool* pool = nullptr;
    int d = 0, d_pad = 0, device = 0, sm_count = 0;
    cudaStream_t stream = nullptr, own_stream = nullptr;
    float* x32 = nullptr;
    __nv_bfloat16* x16 = nullptr;
    VmmApi vmm;                           // in-place growth of x32 / x16 (falls back to cudaMalloc + copy)
    VBuf v32, v16;
    size_t vmm_gran = 0;
    int64_t n = 0, cap_rows = 0, row_offset = 0;
    bool store16 = false;                 // rows ARE 16-bit (bf16 or fp16 per `sh`): no fp32 master
    int sh = SH_BF16;                     // operand type of the coarse GEMM = element type of x16
    unsigned int* norm_stats = nullptr;   // device [2]
    long long* gstats = nullptr;          // device [GS_COUNT]
    long long* h_gstats = nullptr;        // pinned host mirror
    PFN_encodeTiled encode = nullptr;
    // grow-only workspace
    DevBuf q16, eps2, thr, cnt, kept, flags, cand, qstage, qhalf, out_s, out_r, exact_scores, exact_misc,
        qlist, stage, seg_tab, gmax;
    int n_seg = 0;                        // row segments (b2ip_set_row_segments); 0 = row_offset
    std::vector<cudaEvent_t> ev_pool, ev_fin;
    cudaEvent_t ev_t0 = nullptr, ev_t1 = nullptr;
    b2ip_stats_t stats;
    std::string err;
    int gx = 0;                           // x-tiles per raster group; 0 = sm_count / 2
    int hint_q = 0, hint_x = 0;           // 0 normal, 1 evict_first, 2 evict_last
    int dbg = 0;
    int verbose = 0;
    int pair = 1;                         // CTA-pair (cta_group::2) scoring kernel when nq > 128
    int stream_kernel = 1;                // nq <= 64: streaming kernel (corpus on the MMA's M side)
    int list_fill_pct = 70;               // adaptive slab schedule: expected list fill after the next slab (% of cap)
    int bootstrap = 1;                    // nq <= 64: threshold from ONE group-max launch over a corpus sample, then
                                          // one filtered slab over all rows (instead of the geometric slab schedule)
    int bootstrap_max_mb = 64;            // ... while the sample (read twice) is at most this many MiB of 16-bit rows
    int dense_first = 1;                  // first slab stored positionally (no counters / hit extraction)
    int fuse_refresh = 1;                 // last threshold refresh inside the finalize kernel
    int two_stage = 1;                    // finalize rescoring in two stages (window eps instead of 2 eps)
    long long cand_budget_bytes = 6ll << 30;
    CUtensorMap tmap_x, tmap_x_pair;      // cached TMA descriptors of x16 (single / pair box)
    // peer-direct exchange of the current b2ip_search_exchange call (n_extra == 0 otherwise)
    int n_extra = 0;
    char* extra_base[MAX_PEERS - 1] = {};   // peer slots for this rank's results: [rows | scores]
    const b2ip_exchange_t* ex = nullptr;
    unsigned int ex_seq = 0;
    long long ex_prior_overflow = 0;      // overflowed queries of earlier query batches of this search
    float* ex_out_s = nullptr;
    int64_t* ex_out_r = nullptr;
    int extra_rank[MAX_PEERS - 1] = {};     // rank that owns extra_base[e]
    bool ex_thr = false;                    // global threshold round active for this search
    long long ex_timeout_ns = 600ll * 1000000000ll;   // B2IP_EXCHANGE_TIMEOUT_S
    // CUDA-graph replay of small-batch searches (fixed slab schedule): see tensor_search
    int graph = 1;                        // option "graph" / env B2IP_GRAPH
    int graph_timing = 0;                 // keep the per-kernel event records inside the graph (3 us per node:
                                          // off by default; b2ip_stats then reports total_ms only)
    unsigned long long ws_gen = 0;        // bumped when a workspace / row buffer moves
    unsigned long long opt_gen = 0;       // bumped when an option, stream or row mapping changes
    DynArgs* dyn_dev = nullptr;
    DynArgs* dyn_host = nullptr;          // pinned
    struct GraphEntry {
        int64_t nq, n; int k, cap;
        unsigned long long ws_gen, opt_gen;
        bool has_ex; b2ip_exchange_t ex;
        cudaGraphExec_t exec;
        int coarse_launches, total_launches, slabs, sample_rows;
        double coarse_flops;
        size_t ev_used;
        unsigned long long last_use;
    };
    std::vector<GraphEntry> graphs;
    unsigned long long graph_clock = 0;
    long long graph_replays = 0, graph_captures = 0;
    size_t timing_events = 0;             // event triples of the last tensor search (read by b2ip_stats)
    bool timing_pending = false;
    const void* tmap_x_base = nullptr;
    int64_t tmap_x_rows = -1;
};

// A set of handles of ONE process (one per GPU) searched together: b2ip_group_search.
struct b2ip_group_s {
    std::vector<b2ip_handle> hs;
    std::vector<char*> buf;               // per device: [2 x n gather slots | 2 x n x thr_cap floats | 2 flag arrays]
    size_t slot = 0, thr_cap = 0;
    b2ip_exchange_t ex[2][MAX_PEERS];     // [parity][member]
    unsigned int seq = 0;
    std::string err;
    // one persistent worker thread per member
    std::vector<std::thread> th;
    std::mutex m;
    std::condition_variable cv, done;
    std::function<void(int)> job;
    unsigned long long gen = 0;
    int left = 0;
    bool stop = false;
};

namespace {

int fail(b2ip_handle h, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (h) h->err = buf; else g_create_error = buf;
    return code;
}

#define CU_TRY(h, expr)                                                                       \
    do {                                                                                      \
        cudaError_t e__ = (expr);                                                             \
        if (e__ != cudaSuccess) {                                                             \
            cudaGetLastError();                                                               \
            return fail(h, e__ == cudaErrorMemoryAllocation ? B2IP_ERR_OOM : B2IP_ERR_CUDA,   \
                        "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__,    \
                        __LINE__);                                                            \
        }                                                                                     \
    } while (0)

#define RC_TRY(expr)                 \
    do {                             \
        int rc__ = (expr);           \
        if (rc__ != B2IP_OK) return rc__; \
    } while (0)

int ensure(b2ip_handle h, DevBuf& b, size_t bytes) {
    if (b.bytes >= bytes) return B2IP_OK;
    if (b.p) { CU_TRY(h, cudaFree(b.p)); b.p = nullptr; b.bytes = 0; }
    h->ws_gen++;
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&b.p, want);
    if (e != cudaSuccess) { cudaGetLastError(); want = bytes; e = cudaMalloc(&b.p, want); }
    if (e != cudaSuccess) {
        cudaGetLastError();
        b.p = nullptr;
        return fail(h, B2IP_ERR_OOM, "cudaMalloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
    }
    b.bytes = want;
    return B2IP_OK;
}

void release(DevBuf& b) {
    if (b.p) cudaFree(b.p);
    b.p = nullptr;
    b.bytes = 0;
}

template <typename F>
bool vmm_sym(const char* name, F* out) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint(name, &fn, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess || !fn) {
        cudaGetLastError();
        return false;
    }
    *out = reinterpret_cast<F>(fn);
    return true;
}

void vmm_init(b2ip_handle h) {
    VmmApi& a = h->vmm;
    if (const char* e = getenv("B2IP_VMM")) if (atoi(e) == 0) return;
    a.ok = vmm_sym("cuMemGetAllocationGranularity", &a.getGranularity) && vmm_sym("cuMemAddressReserve", &a.addressReserve) &&
           vmm_sym("cuMemCreate", &a.create) && vmm_sym("cuMemMap", &a.map) && vmm_sym("cuMemSetAccess", &a.setAccess) &&
           vmm_sym("cuMemUnmap", &a.unmap) && vmm_sym("cuMemRelease", &a.release) && vmm_sym("cuMemAddressFree", &a.addressFree);
    if (!a.ok) return;
    CUmemAllocationProp prop{};
    prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
    prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    prop.location.id = h->device;
    if (a.getGranularity(&h->vmm_gran, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED) != CUDA_SUCCESS || h->vmm_gran == 0) a.ok = false;
}

// maps physical memory behind [0, bytes) of the buffer (reserving its address range on first use)
bool vmm_grow(b2ip_handle h, VBuf& b, size_t bytes) {
    VmmApi& a = h->vmm;
    if (bytes <= b.mapped) return true;
    if (!b.base) {
        size_t free_b = 0, total_b = 0;
        if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) { cudaGetLastError(); return false; }
        b.reserved = (total_b + h->vmm_gran - 1) / h->vmm_gran * h->vmm_gran;   // a buffer never outgrows the device
        if (a.addressReserve(&b.base, b.reserved, h->vmm_gran, 0, 0) != CUDA_SUCCESS) { b.base = 0; b.reserved = 0; return false; }
    }
    if (bytes > b.reserved) return false;
    // chunks grow geometrically up to 256 MiB: a small index maps a few MiB, a large one few chunks
    const size_t gran = h->vmm_gran;
    const size_t max_step = std::max<size_t>(gran, 256u << 20) / gran * gran;
    while (b.mapped < bytes) {
        size_t step = std::max(bytes - b.mapped, b.mapped / 2);
        step = std::min(max_step, (step + gran - 1) / gran * gran);
        size_t len = std::min<size_t>(step, b.reserved - b.mapped);
        CUmemAllocationProp prop{};
        prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
        prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
        prop.location.id = h->device;
        CUmemGenericAllocationHandle hd;
        if (a.create(&hd, len, &prop, 0) != CUDA_SUCCESS) return false;
        if (a.map(b.base + b.mapped, len, 0, hd, 0) != CUDA_SUCCESS) { a.release(hd); return false; }
        CUmemAccessDesc acc{};
        acc.location = prop.location;
        acc.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
        if (a.setAccess(b.base + b.mapped, len, &acc, 1) != CUDA_SUCCESS) { a.unmap(b.base + b.mapped, len); a.release(hd); return false; }
        b.chunks.emplace_back(hd, len);
        b.mapped += len;
    }
    return true;
}

void vmm_free(b2ip_handle h, VBuf& b) {
    if (!b.base) return;
    size_t off = 0;
    for (auto& c : b.chunks) { h->vmm.unmap(b.base + off, c.second); h->vmm.release(c.first); off += c.second; }
    h->vmm.addressFree(b.base, b.reserved);
    b = VBuf();
}

int grow_rows(b2ip_handle h, int64_t need, bool exact = false) {
    if (need <= h->cap_rows) return B2IP_OK;
    const size_t row32 = static_cast<size_t>(h->d) * sizeof(float), row16 = static_cast<size_t>(h->d_pad) * 2;
    if (h->vmm.ok && (h->n == 0 || h->v16.base)) {
        // in place: the rows keep their addresses, nothing is copied
        const bool first = h->v16.base == 0;
        if (first && (h->x32 || h->x16)) {           // (a cudaMalloc'ed buffer from before: none when n == 0)
            if (h->x32) cudaFree(h->x32);
            if (h->x16) cudaFree(h->x16);
            h->x32 = nullptr; h->x16 = nullptr; h->cap_rows = 0;
        }
        const bool ok = (h->store16 || vmm_grow(h, h->v32, static_cast<size_t>(need) * row32)) &&
                        vmm_grow(h, h->v16, static_cast<size_t>(need) * row16);
        if (ok) {
            h->x32 = h->store16 ? nullptr : reinterpret_cast<float*>(h->v32.base);
            h->x16 = reinterpret_cast<__nv_bfloat16*>(h->v16.base);
            int64_t cap = static_cast<int64_t>(h->v16.mapped / row16);
            if (!h->store16) cap = std::min<int64_t>(cap, static_cast<int64_t>(h->v32.mapped / row32));
            h->cap_rows = cap;
            if (first) h->ws_gen++;
            return B2IP_OK;
        }
        if (h->n > 0 || !first)
            return fail(h, B2IP_ERR_OOM, "growing the index to %lld rows failed (device memory exhausted)",
                        static_cast<long long>(need));
        // nothing stored yet and the very first mapping failed: use plain allocations instead
        vmm_free(h, h->v32);
        vmm_free(h, h->v16);
        h->x32 = nullptr; h->x16 = nullptr; h->cap_rows = 0;
        h->vmm.ok = false;
    }
    int64_t ncap = need;
    if (!exact) ncap = std::max<int64_t>(std::max<int64_t>(need, h->cap_rows + h->cap_rows / 2), 4096);
    float* nx32 = nullptr;
    __nv_bfloat16* nx16 = nullptr;
    auto alloc_both = [&](int64_t rows) {
        cudaError_t e = cudaSuccess;
        if (!h->store16) e = cudaMalloc(&nx32, static_cast<size_t>(rows) * h->d * sizeof(float));
        if (e == cudaSuccess) e = cudaMalloc(&nx16, static_cast<size_t>(rows) * h->d_pad * 2);
        return e;
    };
    cudaError_t e = alloc_both(ncap);
    if (e != cudaSuccess && ncap > need) {   // retry with the exact size
        cudaGetLastError();
        if (nx32) cudaFree(nx32);
        nx32 = nullptr; nx16 = nullptr;
        ncap = need;
        e = alloc_both(ncap);
    }
    if (e != cudaSuccess) {
        cudaGetLastError();
        if (nx32) cudaFree(nx32);
        if (nx16) cudaFree(nx16);
        return fail(h, B2IP_ERR_OOM, "growing the index to %lld rows failed: %s",
                    static_cast<long long>(ncap), cudaGetErrorString(e));
    }
    if (h->n > 0) {
        if (!h->store16)
            CU_TRY(h, cudaMemcpyAsync(nx32, h->x32, static_cast<size_t>(h->n) * h->d * sizeof(float),
                                      cudaMemcpyDeviceToDevice, h->stream));
        CU_TRY(h, cudaMemcpyAsync(nx16, h->x16, static_cast<size_t>(h->n) * h->d_pad * 2,
                                  cudaMemcpyDeviceToDevice, h->stream));
        CU_TRY(h, cudaStreamSynchronize(h->stream));
    }
    if (h->x32) cudaFree(h->x32);
    if (h->x16) cudaFree(h->x16);
    h->x32 = nx32;
    h->x16 = nx16;
    h->cap_rows = ncap;
    h->ws_gen++;
    return B2IP_OK;
}

int make_tmap_bf16(b2ip_handle h, CUtensorMap* m, const void* base, int64_t rows, int d_pad,
                   int box_rows) {
    cuuint64_t dims[2] = {static_cast<cuuint64_t>(d_pad), static_cast<cuuint64_t>(rows)};
    cuuint64_t strides[1] = {static_cast<cuuint64_t>(d_pad) * 2};
    cuuint32_t box[2] = {KBLOCK_ELEMS, static_cast<cuuint32_t>(box_rows)};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = h->encode(m, h->sh == SH_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims,
                           strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS)
        return fail(h, B2IP_ERR_CUDA, "cuTensorMapEncodeTiled failed (CUresult %d, rows=%lld d_pad=%d)",
                    static_cast<int>(r), static_cast<long long>(rows), d_pad);
    return B2IP_OK;
}

unsigned long long hint_policy(int v) {
    return v == 1 ? ptx::kEvictFirst : (v == 2 ? ptx::kEvictLast : ptx::kEvictNormal);
}

cudaEvent_t get_event(std::vector<cudaEvent_t>& pool, size_t i) {
    while (pool.size() <= i) {
        cudaEvent_t e;
        cudaEventCreate(&e);
        pool.push_back(e);
    }
    return pool[i];
}
cudaEvent_t get_event(b2ip_handle h, size_t i) { return get_event(h->ev_pool, i); }

// finalize_kernel<true>: [sort buffer | query fp32 | per-warp ring of `stages` rows | mbarriers]
int rescore_ring_stages(b2ip_handle h) {
    // ~64 KB of rows in flight per CTA (8 warps x stages x row): three CTAs per SM
    const size_t row_bytes = h->store16 ? static_cast<size_t>(h->d_pad) * 2 : static_cast<size_t>(h->d) * 4;
    const size_t nw = SEL_THREADS / 32;
    size_t ns = std::max<size_t>(2, std::min<size_t>(8, (64u << 10) / (nw * row_bytes)));
    while (ns > 1 && nw * ns * (row_bytes + 8) + static_cast<size_t>(h->d) * 4 + 64 > (200u << 10)) ns--;
    return static_cast<int>(ns);
}
size_t finalize_smem_bytes(b2ip_handle h, int stages) {
    const size_t row_bytes = h->store16 ? static_cast<size_t>(h->d_pad) * 2 : static_cast<size_t>(h->d) * 4;
    const size_t nw = SEL_THREADS / 32;
    const size_t uni = std::max<size_t>(SORT_CAP * sizeof(unsigned long long), nw * stages * row_bytes);
    return uni + ((static_cast<size_t>(h->d) * 4 + 15) & ~static_cast<size_t>(15)) + nw * stages * 8;
}

int64_t pad_q(int64_t nq) { return (nq + 2 * TILE_Q - 1) / (2 * TILE_Q) * (2 * TILE_Q); }

// ------------------------------------------------------------------------- host -> device staging
// Worker threads that copy one host range in parallel slices (pageable -> pinned).
class CopyPool {
  public:
    explicit CopyPool(int n) : n_(n) {
        for (int i = 0; i < n; i++) th_.emplace_back([this, i] { run(i); });
    }
    ~CopyPool() {
        { std::lock_guard<std::mutex> l(m_); stop_ = true; gen_++; }
        cv_.notify_all();
        for (auto& t : th_) t.join();
    }
    void copy(void* dst, const void* src, size_t bytes) {
        if (n_ == 0 || bytes < (1u << 20)) { memcpy(dst, src, bytes); return; }
        std::unique_lock<std::mutex> l(m_);
        dst_ = static_cast<char*>(dst); src_ = static_cast<const char*>(src); bytes_ = bytes;
        left_ = n_; gen_++;
        cv_.notify_all();
        done_.wait(l, [this] { return left_ == 0; });
    }
  private:
    void run(int i) {
        int seen = 0;
        std::unique_lock<std::mutex> l(m_);
        for (;;) {
            cv_.wait(l, [&] { return gen_ != seen; });
            seen = gen_;
            if (stop_) return;
            char* d = dst_; const char* s = src_; const size_t b = bytes_;
            l.unlock();
            size_t per = (b + n_ - 1) / n_;
            per = (per + 4095) & ~static_cast<size_t>(4095);
            const size_t o = per * static_cast<size_t>(i);
            if (o < b) memcpy(d + o, s + o, std::min(per, b - o));
            l.lock();
            if (--left_ == 0) done_.notify_one();
        }
    }
    int n_;
    std::vector<std::thread> th_;
    std::mutex m_;
    std::condition_variable cv_, done_;
    char* dst_ = nullptr; const char* src_ = nullptr; size_t bytes_ = 0;
    int left_ = 0, gen_ = 0;
    bool stop_ = false;
};

constexpr size_t PIN_CHUNK_BYTES = 16u << 20;        // two pinned staging buffers of this size
constexpr int64_t INGEST_CHUNK_BYTES = 64ll << 20;   // rows landed / converted per step

// dst (device) <- src (host), ordered on the handle's stream.  Page-locked sources go straight
// to the copy engine; pageable ones through two pinned buffers filled by the CopyPool, so the
// CPU copy of piece i+1 overlaps the DMA of piece i (the driver's own pageable path: ~11 GB/s).
int ensure_pinned_staging(b2ip_handle h) {
    if (h->pin[0]) return B2IP_OK;
    for (int b = 0; b < 2; b++) {
        CU_TRY(h, cudaHostAlloc(&h->pin[b], PIN_CHUNK_BYTES, cudaHostAllocDefault));
        CU_TRY(h, cudaEventCreateWithFlags(&h->pin_ev[b], cudaEventDisableTiming));
    }
    int nt = 4;
    if (const char* s = getenv("B2IP_COPY_THREADS")) nt = std::max(0, std::min(32, atoi(s)));
    h->pool = new CopyPool(nt);
    return B2IP_OK;
}

int host_to_device(b2ip_handle h, void* dst, const void* src, size_t bytes) {
    cudaPointerAttributes attr;
    bool pinned = cudaPointerGetAttributes(&attr, src) == cudaSuccess && attr.type != cudaMemoryTypeUnregistered;
    cudaGetLastError();
    if (pinned || bytes < (256u << 10)) {
        CU_TRY(h, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, h->stream));
        return B2IP_OK;
    }
    RC_TRY(ensure_pinned_staging(h));
    for (size_t off = 0; off < bytes; off += PIN_CHUNK_BYTES) {
        const size_t len = std::min(PIN_CHUNK_BYTES, bytes - off);
        const int b = h->pin_next;
        h->pin_next ^= 1;
        CU_TRY(h, cudaEventSynchronize(h->pin_ev[b]));      // the DMA that last read this buffer is done
        h->pool->copy(h->pin[b], static_cast<const char*>(src) + off, len);
        CU_TRY(h, cudaMemcpyAsync(static_cast<char*>(dst) + off, h->pin[b], len, cudaMemcpyHostToDevice, h->stream));
        CU_TRY(h, cudaEventRecord(h->pin_ev[b], h->stream));
    }
    return B2IP_OK;
}

int ensure_pinned_staging(b2ip_handle h);

// dst (host) <- src (device); complete on return.  Pageable destinations are filled from the
// two pinned buffers, the CPU copy of piece i overlapping the DMA of piece i+1.
int device_to_host(b2ip_handle h, void* dst, const void* src, size_t bytes) {
    cudaPointerAttributes attr;
    bool pinned = cudaPointerGetAttributes(&attr, dst) == cudaSuccess && attr.type != cudaMemoryTypeUnregistered;
    cudaGetLastError();
    if (pinned || bytes < (256u << 10)) {
        CU_TRY(h, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, h->stream));
        CU_TRY(h, cudaStreamSynchronize(h->stream));
        return B2IP_OK;
    }
    RC_TRY(ensure_pinned_staging(h));
    CU_TRY(h, cudaEventSynchronize(h->pin_ev[0]));
    CU_TRY(h, cudaEventSynchronize(h->pin_ev[1]));
    size_t prev_off = 0, prev_len = 0;
    int prev_b = -1;
    for (size_t off = 0; off < bytes; off += PIN_CHUNK_BYTES) {
        const size_t len = std::min(PIN_CHUNK_BYTES, bytes - off);
        const int b = h->pin_next;
        h->pin_next ^= 1;
        CU_TRY(h, cudaMemcpyAsync(h->pin[b], static_cast<const char*>(src) + off, len, cudaMemcpyDeviceToHost, h->stream));
        CU_TRY(h, cudaEventRecord(h->pin_ev[b], h->stream));
        if (prev_b >= 0) {
            CU_TRY(h, cudaEventSynchronize(h->pin_ev[prev_b]));
            h->pool->copy(static_cast<char*>(dst) + prev_off, h->pin[prev_b], prev_len);
        }
        prev_b = b; prev_off = off; prev_len = len;
    }
    if (prev_b >= 0) {
        CU_TRY(h, cudaEventSynchronize(h->pin_ev[prev_b]));
        h->pool->copy(static_cast<char*>(dst) + prev_off, h->pin[prev_b], prev_len);
    }
    return B2IP_OK;
}

struct Guard {   // selects the index's device for the duration of a call
    int prev = -1;
    explicit Guard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
    ~Guard() { if (prev >= 0) cudaSetDevice(prev); }
};

// ------------------------------------------------------------------------- exact path
// Scores qlist's queries (indices into q32) against the whole shard in fp32 and writes their
// top-k.  qlist_dev == nullptr means queries [q_begin, q_begin + nql).
int exact_search(b2ip_handle h, const float* q32, const int* qlist_host, int64_t nql, int k,
                 float* d_scores, int64_t* d_rows) {
    const int64_t n = h->n;
    RC_TRY(ensure(h, h->exact_scores, static_cast<size_t>(EXACT_QB) * n * sizeof(float)));
    const size_t misc_bytes = sizeof(ExactState) + EXACT_QB * 256 * sizeof(unsigned int) +
                              EXACT_QB * sizeof(int) + 64;
    RC_TRY(ensure(h, h->exact_misc, misc_bytes));
    RC_TRY(ensure(h, h->qlist, static_cast<size_t>(nql) * sizeof(int)));
    const int cap = k;
    RC_TRY(ensure(h, h->cand, static_cast<size_t>(EXACT_QB) * cap * sizeof(unsigned long long)));
    auto* st = reinterpret_cast<ExactState*>(h->exact_misc.p);
    auto* ghist = reinterpret_cast<unsigned int*>(reinterpret_cast<char*>(h->exact_misc.p) + sizeof(ExactState));
    int* gcnt = reinterpret_cast<int*>(ghist + EXACT_QB * 256);
    int* qlist_dev = reinterpret_cast<int*>(h->qlist.p);
    CU_TRY(h, cudaMemcpyAsync(qlist_dev, qlist_host, static_cast<size_t>(nql) * sizeof(int),
                              cudaMemcpyHostToDevice, h->stream));
    const size_t sq_bytes = static_cast<size_t>(EXACT_QB) * h->d * sizeof(float);
    const size_t fin_smem = SORT_CAP * sizeof(unsigned long long);     // finalize_kernel<false>: sort only
    const int sgrid = static_cast<int>(std::min<int64_t>((n + 7) / 8, static_cast<int64_t>(h->sm_count) * 8));
    const int hgrid = static_cast<int>(std::min<int64_t>((n + 255) / 256, static_cast<int64_t>(h->sm_count) * 4));
    for (int64_t g0 = 0; g0 < nql; g0 += EXACT_QB) {
        const int nqg = static_cast<int>(std::min<int64_t>(EXACT_QB, nql - g0));
        exact_scores_kernel<<<std::max(sgrid, 1), 256, sq_bytes, h->stream>>>(
            h->x32, h->x16, n, h->d, h->d_pad, h->sh, q32, qlist_dev + g0, nqg,
            reinterpret_cast<float*>(h->exact_scores.p));
        exact_init_kernel<<<1, 256, 0, h->stream>>>(st, ghist, gcnt, k);
        for (int pass = 0; pass < 8; pass++) {
            exact_hist_kernel<<<dim3(std::max(hgrid, 1), nqg), 256, 0, h->stream>>>(
                reinterpret_cast<float*>(h->exact_scores.p), n, pass, st, ghist);
            exact_pick_kernel<<<nqg, 32, 0, h->stream>>>(st, ghist, pass);
        }
        exact_collect_kernel<<<dim3(std::max(hgrid, 1), nqg), 256, 0, h->stream>>>(
            reinterpret_cast<float*>(h->exact_scores.p), n, st,
            reinterpret_cast<unsigned long long*>(h->cand.p), gcnt, cap);
        FinalizeParams fp{};
        fp.k = k; fp.cap = cap; fp.d = h->d;
        fp.qlist = qlist_dev + g0;
        fp.cand = reinterpret_cast<unsigned long long*>(h->cand.p);
        fp.cnt = gcnt; fp.flags = nullptr; fp.q32 = q32; fp.x32 = h->x32;
        fp.x16 = h->x16; fp.d_pad = h->d_pad; fp.sh = h->sh;
        fp.row_offset = h->row_offset;
        fp.n_seg = h->n_seg;
        fp.seg_local = static_cast<const long long*>(h->seg_tab.p);
        fp.seg_delta = fp.seg_local + h->n_seg;
        fp.out_scores = d_scores; fp.out_rows = reinterpret_cast<long long*>(d_rows);
        fp.gstats = nullptr;
        fp.n_extra = 0;
        finalize_kernel<false><<<nqg, SEL_THREADS, fin_smem, h->stream>>>(fp);
        h->stats.total_launches += 20;
    }
    CU_TRY(h, cudaGetLastError());
    return B2IP_OK;
}

// ------------------------------------------------------------------------- peer-direct exchange
// After the last finalize of a search: tell every rank that this rank's [nq,k] block is in its
// memory, then merge the world's blocks out of THIS rank's gather buffer as soon as all flags are
// in.  Two launches behind finalize on the same stream -- no host round trip, no NCCL call.
PeerFlags peer_flags(const b2ip_exchange_t* ex) {
    PeerFlags pf{};
    pf.world = ex->world;
    pf.rank = ex->rank;
    for (int p = 0; p < ex->world; p++) pf.flags[p] = static_cast<unsigned int*>(ex->flags[p]);
    return pf;
}

// queries [q_lo, q_hi) of a search of nq queries belong to `rank` in owner mode
void owner_range(const b2ip_exchange_t* ex, int64_t nq, int64_t* q_lo, int64_t* q_hi, int64_t* per) {
    *per = (nq + ex->world - 1) / ex->world;
    *q_lo = std::min<int64_t>(static_cast<int64_t>(ex->rank) * *per, nq);
    *q_hi = std::min<int64_t>(*q_lo + *per, nq);
}

int enqueue_exchange(b2ip_handle h, int64_t nq, int k, const DynArgs* dyn = nullptr) {
    const b2ip_exchange_t* ex = h->ex;
    exchange_signal_kernel<<<1, 32, 0, h->stream>>>(peer_flags(ex), h->ex_seq, XF_RESULT, h->gstats,
                                                    h->ex_prior_overflow, dyn);
    h->stats.total_launches += 1;
    int P = 2;
    while (P < ex->world * k) P <<= 1;
    const size_t smem = static_cast<size_t>(P) * sizeof(unsigned long long);
    if (smem > 200 * 1024) return fail(h, B2IP_ERR_UNSUPPORTED, "exchange: world*k=%d too large", ex->world * k);
    CU_TRY(h, cudaFuncSetAttribute(merge_topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    int64_t q_lo = 0, q_hi = nq, per = 0;
    if (ex->gather_mode == B2IP_GATHER_OWNER) owner_range(ex, nq, &q_lo, &q_hi, &per);
    const char* mine = static_cast<const char*>(ex->gather[ex->rank]);
    // (a rank that owns no query still has to run the signal above; its merge is empty.  The wait
    // for the peers' flags and the status word then happen in a 1-CTA launch over zero queries.)
    const unsigned int grid = static_cast<unsigned int>(std::max<int64_t>(q_hi - q_lo, 0));
    if (grid > 0) {
        merge_topk_kernel<<<grid, SEL_THREADS, smem, h->stream>>>(
            nq, k, ex->world, reinterpret_cast<const float*>(mine + static_cast<size_t>(nq) * k * 8),
            reinterpret_cast<const long long*>(mine), ex->slot_bytes / 4, ex->slot_bytes / 8, h->ex_out_s,
            reinterpret_cast<long long*>(h->ex_out_r), P, static_cast<const unsigned int*>(ex->flags[ex->rank]),
            h->ex_seq, h->gstats + GS_XSTATUS, q_lo, h->ex_timeout_ns, dyn);
    } else {
        exchange_wait_kernel<<<1, 32, 0, h->stream>>>(static_cast<const unsigned int*>(ex->flags[ex->rank]),
                                                      ex->world, h->ex_seq, h->gstats + GS_XSTATUS, h->ex_timeout_ns, dyn);
    }
    h->stats.total_launches += 1;
    return B2IP_OK;
}

// ------------------------------------------------------------------------- tensor path
// Sample of the threshold bootstrap (see tensor_search): *grid CTAs over *tiles tiles of 128 rows, or
// *grid = 0 when the batch keeps the geometric schedule.  Pure host arithmetic (also reachable as
// b2ip_debug_plan_bootstrap, so the CPU test suite can sweep it without a GPU).
void plan_bootstrap(int64_t n, int k, int cap, int sm_count, int d_pad, int max_mb, int* grid, int64_t* tiles) {
    *grid = 0;
    *tiles = 0;
    if (n <= 0 || k < 1 || cap < 1 || sm_count < 1) return;
    // full tiles only (every group holds a row), the sample at most 1/16 of the corpus, and
    // >= 16 groups per wanted result (two of the k best rows rarely share a group)
    const int64_t tiles_all = (n + STREAM_TILE_X - 1) / STREAM_TILE_X;
    const int boot_grid = static_cast<int>(std::min<int64_t>(std::min<int64_t>(sm_count, BOOT_MAX_GROUPS / STREAM_TILE_X),
                                                             (tiles_all - 1) / 16));
    if (boot_grid < 1 || static_cast<int64_t>(boot_grid) * STREAM_TILE_X < 16ll * k) return;
    const int64_t want_rows = (6ll * k * n + cap - 1) / cap;
    int64_t boot_tiles = std::max<int64_t>(boot_grid, (want_rows + STREAM_TILE_X - 1) / STREAM_TILE_X);
    // the launch lasts as long as its busiest CTA: a few tiles past a whole wave are not worth
    // another round (2,625,000 rows: 301 tiles -> 296 = 2 per SM; the sample shrinks by < 1/8 wave)
    if (boot_tiles > boot_grid && boot_tiles % boot_grid < boot_grid / 8) boot_tiles -= boot_tiles % boot_grid;
    // ... and only while reading the sample twice costs less than the two launch + refresh
    // rounds it replaces (~45 us): option bootstrap_max_mb (16-bit bytes of the sample).
    // At d = 768, k = 10 that is a shard of up to ~3M rows -- one GPU of eight on the 21M-row
    // corpus; a whole-corpus GPU keeps the geometric schedule (measured: DESIGN 4.1e)
    const int64_t sample_bytes = boot_tiles * STREAM_TILE_X * d_pad * 2;
    if (boot_tiles * 16 > tiles_all - 1 || sample_bytes > (static_cast<int64_t>(max_mb) << 20)) return;
    *grid = boot_grid;
    *tiles = boot_tiles;
}

int tensor_search(b2ip_handle h, const float* q32, int64_t nq, int k, float* d_scores,
                  int64_t* d_rows) {
    const int64_t n = h->n;
    // List capacity: lists of <= 4096 keys are refreshed / finalized entirely in shared memory
    // (REFRESH_SMEM_KEYS, SORT_CAP), so k <= 1024 keeps that size and pays with a few more slabs
    // (measured at k = 1000: refresh + finalize 12 % of the step with 16k-key lists selected out of L2)
    const int cap = std::max(4096, 4 * k);
    int64_t qb_max = h->cand_budget_bytes / (static_cast<int64_t>(cap) * 8);
    qb_max = std::max<int64_t>(TILE_Q, qb_max / TILE_Q * TILE_Q);
    const int64_t qb = std::min<int64_t>(nq, qb_max);

    // query rows are padded to whole (pair) tiles with zero rows: a TMA box that hangs over
    // the end of the tensor is served by the (slower) out-of-bounds fill path
    RC_TRY(ensure(h, h->q16, static_cast<size_t>(pad_q(qb)) * h->d_pad * 2));
    RC_TRY(ensure(h, h->eps2, qb * sizeof(float)));
    RC_TRY(ensure(h, h->thr, qb * sizeof(float)));
    RC_TRY(ensure(h, h->cnt, qb * sizeof(int)));
    RC_TRY(ensure(h, h->kept, qb * sizeof(int)));
    RC_TRY(ensure(h, h->flags, qb * sizeof(int)));
    RC_TRY(ensure(h, h->cand, static_cast<size_t>(qb) * cap * 8));

    const int ring_stages = rescore_ring_stages(h);
    const size_t fin_smem = finalize_smem_bytes(h, ring_stages);
    // tensor maps of the corpus are rebuilt only when the rows moved or grew
    if (h->tmap_x_base != h->x16 || h->tmap_x_rows != n) {
        RC_TRY(make_tmap_bf16(h, &h->tmap_x_pair, h->x16, n, h->d_pad, 128));
        RC_TRY(make_tmap_bf16(h, &h->tmap_x, h->x16, n, h->d_pad, TILE_X));
        h->tmap_x_base = h->x16;
        h->tmap_x_rows = n;
    }
    const CUtensorMap& tmap_x_pair = h->tmap_x_pair;
    const CUtensorMap& tmap_x = h->tmap_x;

    // global threshold round of the peer-direct exchange: one query batch only (the flag carries
    // one sequence number per search); every rank takes the same decision (same nq, k, budget)
    // -- and not in the latency regime (nq <= 2048): there the extra flag round (one more launch,
    // one more cross-rank wait) costs more than rescoring a few dozen rows per query less
    const bool thr_round = h->ex && h->ex->gthr[0] && nq <= qb && h->ex->thr_stride >= nq && nq > 2048;
    h->ex_thr = thr_round;
    const bool fuse_refresh = h->fuse_refresh && !thr_round;
    size_t ev_used = 0;
    std::vector<int> fallback;

    // ---- CUDA-graph replay (latency regime) -------------------------------------------------
    // A small batch runs a FIXED launch sequence (prep, slabs + refreshes, finalize, exchange,
    // counters D2H) with no host decision in between: it is captured once per shape and replayed
    // with one cudaGraphLaunch; what differs from call to call travels through DynArgs.
    bool use_graph = false;
    {
        int64_t slab0 = std::min<int64_t>(cap, std::max<int64_t>(1024, 8ll * k)) / TILE_X * TILE_X;
        use_graph = h->graph && !h->verbose && !h->dbg && nq <= qb && nq <= 2048 && n > slab0;
    }
    const DynArgs* dyn = nullptr;
    b2ip_index_s::GraphEntry* entry = nullptr;
    bool capturing = false;
    if (use_graph) {
        DynArgs da{};
        da.q32 = q32; da.out_s = d_scores; da.out_r = reinterpret_cast<long long*>(d_rows);
        da.ex_out_s = h->ex_out_s; da.ex_out_r = reinterpret_cast<long long*>(h->ex_out_r);
        da.seq = h->ex_seq;
        *h->dyn_host = da;
        CU_TRY(h, cudaMemcpyAsync(h->dyn_dev, h->dyn_host, sizeof(DynArgs), cudaMemcpyHostToDevice, h->stream));
        dyn = h->dyn_dev;
        for (auto& ge : h->graphs) {
            if (ge.nq == nq && ge.n == n && ge.k == k && ge.cap == cap && ge.ws_gen == h->ws_gen &&
                ge.opt_gen == h->opt_gen && ge.has_ex == (h->ex != nullptr) &&
                (!h->ex || memcmp(&ge.ex, h->ex, sizeof(b2ip_exchange_t)) == 0)) {
                entry = &ge;
                break;
            }
        }
        if (entry) {
            entry->last_use = ++h->graph_clock;
            h->graph_replays++;
            CU_TRY(h, cudaGraphLaunch(entry->exec, h->stream));
            h->stats.query_batches = 1;
            h->stats.coarse_launches = entry->coarse_launches;
            h->stats.total_launches = entry->total_launches;
            h->stats.slabs = entry->slabs;
            h->stats.sample_rows = entry->sample_rows;
            h->stats.coarse_flops = entry->coarse_flops;
            h->stats.graph_mode = 2;
            ev_used = entry->ev_used;
        } else {
            CU_TRY(h, cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeRelaxed));
            capturing = true;
        }
    }
    // event records: plain outside a graph; inside a capture they become event-record NODES
    // (cudaEventRecordExternal) so the per-kernel times stay measurable, or are left out
    auto rec = [&](cudaEvent_t e) -> cudaError_t {
        if (!capturing) return cudaEventRecord(e, h->stream);
        if (!h->graph_timing) return cudaSuccess;
        return cudaEventRecordWithFlags(e, h->stream, cudaEventRecordExternal);
    };
    // leaves capture mode on an error path
    auto abort_capture = [&]() {
        if (!capturing) return;
        cudaGraph_t g = nullptr;
        cudaStreamEndCapture(h->stream, &g);
        if (g) cudaGraphDestroy(g);
        cudaGetLastError();
        capturing = false;
    };
#define CAP_TRY(expr) do { cudaError_t cap_e__ = (expr); if (cap_e__ != cudaSuccess) { abort_capture(); CU_TRY(h, cap_e__); } } while (0)
#define CAP_RC(expr) do { int rc__ = (expr); if (rc__ != B2IP_OK) { abort_capture(); return rc__; } } while (0)

    for (int64_t q0 = 0; q0 < nq; q0 += qb) {
        const int nqb = static_cast<int>(std::min<int64_t>(qb, nq - q0));
        if (!entry) {
        h->stats.query_batches++;
        const float* qptr = q32 + q0 * h->d;
        const int nq_pad = static_cast<int>(pad_q(nqb));
        // first slab: every row is a candidate (no threshold yet) and is stored at its own
        // position in the list, so the fill counters start at the slab size
        int64_t slab = std::min<int64_t>(cap, std::max<int64_t>(1024, 8ll * k));
        slab = slab / TILE_X * TILE_X;
        const int64_t first_slab = std::min<int64_t>(slab, n);
        const bool dense_first = h->dense_first != 0;
        CUtensorMap tmap_q;
        CAP_RC(make_tmap_bf16(h, &tmap_q, h->q16.p, pad_q(nqb), h->d_pad, TILE_Q));
        const bool use_pair = h->pair && nqb > TILE_Q && h->sm_count >= 2;
        // small batches: streaming kernel (corpus tile on the M side, resident queries) when the
        // padded batch fits next to at least 4 corpus stages in shared memory
        const int nq_s = nqb <= 32 ? 32 : 64;
        const size_t q_bytes = static_cast<size_t>(h->d_pad / KBLOCK_ELEMS) * nq_s * KBLOCK_BYTES;
        const int stages = static_cast<int>(std::min<long long>(
            STREAM_STAGES, (static_cast<long long>(MAX_SMEM_OPTIN) - STREAM_MISC_BYTES - static_cast<long long>(q_bytes)) / STREAM_X_STAGE_BYTES));
        const bool use_stream = h->stream_kernel && nqb <= 64 && stages >= 4;
        const size_t stream_smem = static_cast<size_t>(std::max(stages, 0)) * STREAM_X_STAGE_BYTES + q_bytes + STREAM_MISC_BYTES;
        if (use_stream) CAP_RC(make_tmap_bf16(h, &tmap_q, h->q16.p, pad_q(nqb), h->d_pad, nq_s));
        // Threshold bootstrap (latency regime, streaming kernel): the geometric schedule spends two
        // dependent rounds (dense slab -> refresh -> small slab -> refresh) before the main slab may
        // start.  Instead: ONE group-max launch over a sample of boot_tiles tiles spread evenly
        // over the corpus (boot_grid CTAs; see coarse_stream_kernel<NQ, true>), the
        // k-th largest group maximum becomes the threshold, and one filtered slab then covers ALL
        // rows.  Sample size: the same margin as the geometric schedule -- k * n / sample_rows, the
        // expected number of rows above the sample's k-th score, is cap / 6: the threshold lies
        // 2 eps below that score (measured on the benchmark's corpus: x1.5 - x2 more rows at k = 10)
        // and the k-th order statistic of a sample is noisy (+-32 % at k = 10; a batch of 64 sees
        // +2.5 sigma).  The sample is read twice, so the bootstrap is only taken when it is a small
        // part of the corpus (k <= 42 at the default capacity).
        int boot_grid = 0;
        int64_t boot_tiles = 0;
        if (use_stream && h->bootstrap && !h->dbg && n > slab)
            plan_bootstrap(n, k, cap, h->sm_count, h->d_pad, h->bootstrap_max_mb, &boot_grid, &boot_tiles);
        const bool bootstrap = boot_grid > 0;
        if (bootstrap) CAP_RC(ensure(h, h->gmax, static_cast<size_t>(nq_s) * boot_grid * STREAM_TILE_X * sizeof(uint32_t)));
        prep_queries_kernel<<<(nq_pad + 7) / 8, 256, 0, h->stream>>>(
            qptr, reinterpret_cast<__nv_bfloat16*>(h->q16.p), nqb, h->d, h->d_pad, h->norm_stats,
            reinterpret_cast<float*>(h->eps2.p), reinterpret_cast<float*>(h->thr.p),
            reinterpret_cast<int*>(h->cnt.p), reinterpret_cast<int*>(h->kept.p),
            reinterpret_cast<int*>(h->flags.p), h->sh, nq_pad, h->gstats,
            dense_first && !bootstrap ? static_cast<int>(first_slab) : 0, dyn);
        h->stats.total_launches++;

        CoarseParams cp{};
        cp.num_k_blocks = h->d_pad / KBLOCK_ELEMS;
        cp.q_tiles = use_pair ? (nqb + 2 * TILE_Q - 1) / (2 * TILE_Q) : (nqb + TILE_Q - 1) / TILE_Q;
        cp.gx = h->gx;
        cp.nq = nqb;
        cp.thr = reinterpret_cast<float*>(h->thr.p);
        cp.cand = reinterpret_cast<unsigned long long*>(h->cand.p);
        cp.cnt = reinterpret_cast<int*>(h->cnt.p);
        cp.cap = cap;
        cp.dump = nullptr;
        cp.dump_ld = 0;
        cp.hint_q = hint_policy(h->hint_q);
        cp.hint_x = hint_policy(h->hint_x);
        cp.dbg = h->dbg;
        cp.idesc = use_pair ? IDESC_PAIR[h->sh] : IDESC_SINGLE[h->sh];
        if (use_stream) cp.idesc = ptx::umma_idesc(h->sh == SH_F16 ? 0 : 1, STREAM_TILE_X, nq_s);

        int64_t done = 0;
        long long overflowed = 0;
        // Latency regime (small query batches): a FIXED geometric slab schedule, no host
        // round-trip between slabs.  Growth r is chosen so that ~3k*r expected new hits stay below
        // half the list capacity; a list that overflows anyway sends its query to the exact path.
        const bool fixed_schedule = nqb <= 2048 && n > slab && !bootstrap;
        double growth = 0.0;
        if (fixed_schedule) {
            const double r_max = std::max(2.0, 0.5 * cap / (3.0 * k));
            const double span = static_cast<double>(n) / static_cast<double>(slab);
            const int steps = std::max(1, static_cast<int>(std::ceil(std::log(span) / std::log(r_max))));
            growth = std::pow(span, 1.0 / steps);
        }
        if (bootstrap) {
            const int64_t boot_rows = boot_tiles * STREAM_TILE_X;
            cp.x_row0 = 0;
            cp.x_row_end = n;
            cp.x_tiles = static_cast<int>(boot_tiles);
            // tile t of the sample = rows [t * gstride, +128): the last one ends before the last full tile does
            cp.gstride = (n / STREAM_TILE_X) / cp.x_tiles * STREAM_TILE_X;
            cp.dense = 0;
            cp.gmax = reinterpret_cast<uint32_t*>(h->gmax.p);
            cudaEvent_t e0 = get_event(h, ev_used++), e1 = get_event(h, ev_used++), e2 = get_event(h, ev_used++);
            CAP_TRY(rec(e0));
            if (nq_s == 32)
                coarse_stream_kernel<32, true><<<boot_grid, COARSE_THREADS, stream_smem, h->stream>>>(
                    tmap_q, tmap_x_pair, cp, stages);
            else
                coarse_stream_kernel<64, true><<<boot_grid, COARSE_THREADS, stream_smem, h->stream>>>(
                    tmap_q, tmap_x_pair, cp, stages);
            CAP_TRY(rec(e1));
            bootstrap_threshold_kernel<<<nqb, SEL_THREADS, static_cast<size_t>(boot_grid) * STREAM_TILE_X * sizeof(uint32_t), h->stream>>>(
                reinterpret_cast<const uint32_t*>(h->gmax.p), boot_grid * STREAM_TILE_X, k,
                reinterpret_cast<float*>(h->thr.p), reinterpret_cast<const float*>(h->eps2.p));
            CAP_TRY(rec(e2));
            h->stats.coarse_launches++;
            h->stats.total_launches += 2;
            h->stats.slabs++;
            h->stats.coarse_flops += 2.0 * nqb * static_cast<double>(boot_rows) * h->d;
            h->stats.sample_rows = static_cast<int32_t>(boot_rows);
            slab = n;                    // the one filtered slab: every row, the sample included
        }
        while (done < n) {
            int64_t s = std::min<int64_t>(slab, n - done);
            // the kernels index tiles with 32-bit integers: keep q_tiles * x_tiles below 2^30
            // (only reachable with hundreds of millions of short rows per shard)
            s = std::min<int64_t>(s, std::max<int64_t>(1, (1ll << 30) / std::max(1, cp.q_tiles)) * STREAM_TILE_X);
            if (done + s < n) s = std::max<int64_t>(TILE_X, s / TILE_X * TILE_X);
            s = std::min<int64_t>(s, n - done);
            cp.x_row0 = done;
            cp.x_row_end = done + s;
            cp.x_tiles = use_stream ? static_cast<int>((s + STREAM_TILE_X - 1) / STREAM_TILE_X)
                                    : static_cast<int>((s + TILE_X - 1) / TILE_X);
            cp.dense = (done == 0 && dense_first && !bootstrap) ? 1 : 0;
            const bool last = done + s >= n;
            const long long tiles = static_cast<long long>(cp.q_tiles) * cp.x_tiles;
            cudaEvent_t e0 = get_event(h, ev_used++), e1 = get_event(h, ev_used++);
            CAP_TRY(rec(e0));
            if (use_stream) {
                const int grid = static_cast<int>(std::min<long long>(cp.x_tiles, h->sm_count));
                if (nq_s == 32)
                    coarse_stream_kernel<32><<<grid, COARSE_THREADS, stream_smem, h->stream>>>(
                        tmap_q, tmap_x_pair, cp, stages);
                else
                    coarse_stream_kernel<64><<<grid, COARSE_THREADS, stream_smem, h->stream>>>(
                        tmap_q, tmap_x_pair, cp, stages);
            } else if (use_pair) {
                const int grid = 2 * static_cast<int>(std::min<long long>(tiles, h->sm_count / 2));
                coarse_filter_pair_kernel<<<grid, COARSE_THREADS, PAIR_SMEM_BYTES, h->stream>>>(
                    tmap_q, tmap_x_pair, cp);
            } else {
                const int grid = static_cast<int>(std::min<long long>(tiles, h->sm_count));
                coarse_filter_kernel<false><<<grid, COARSE_THREADS, COARSE_SMEM_BYTES, h->stream>>>(
                    tmap_q, tmap_x, cp);
            }
            CAP_TRY(rec(e1));
            // the refresh after the LAST slab is fused into the finalize kernel -- unless this
            // rank owes its peers a bound for the global threshold (it must exist before finalize)
            const bool fused = last && fuse_refresh;
            if (!fused) {
                PublishBound pub{};
                if (last && thr_round) {
                    pub.m_rank = (k + h->ex->world - 1) / h->ex->world;
                    pub.n_dst = h->ex->world;
                    for (int r = 0; r < h->ex->world; r++)
                        pub.dst[r] = static_cast<float*>(h->ex->gthr[r]) + static_cast<size_t>(h->ex->rank) * h->ex->thr_stride + q0;
                }
                refresh_threshold_kernel<<<nqb, SEL_THREADS, 0, h->stream>>>(
                    k, cap, cp.cand, cp.cnt, reinterpret_cast<int*>(h->kept.p),
                    reinterpret_cast<float*>(h->thr.p), reinterpret_cast<float*>(h->eps2.p),
                    reinterpret_cast<int*>(h->flags.p), h->gstats, pub);
            }
            cudaEvent_t e2 = get_event(h, ev_used++);
            CAP_TRY(rec(e2));
            h->stats.coarse_launches++;
            h->stats.total_launches += fused ? 1 : 2;
            h->stats.slabs++;
            h->stats.coarse_flops += 2.0 * nqb * static_cast<double>(s) * h->d;
            done += s;
            if (last) break;
            if (fixed_schedule) {
                slab = std::max<int64_t>(TILE_X, static_cast<int64_t>(static_cast<double>(done) * (growth - 1.0)));
                if (n - done - slab < slab / 4) slab = n - done;          // no tiny tail slab
                continue;
            }
            CU_TRY(h, cudaMemcpyAsync(h->h_gstats, h->gstats, GS_COUNT * sizeof(long long),
                                      cudaMemcpyDeviceToHost, h->stream));
            CU_TRY(h, cudaStreamSynchronize(h->stream));
            CU_TRY(h, cudaGetLastError());
            const long long m_max = std::max<long long>(h->h_gstats[GS_MAX_KEPT], 1);
            overflowed = h->h_gstats[GS_OVERFLOW];
            if (h->verbose) {
                float ms = 0.f;
                cudaEventElapsedTime(&ms, e0, e1);
                fprintf(stderr, "[b2ip] slab rows [%lld,+%lld) %.3f ms %.0f TFLOP/s  max_kept=%lld cand_total=%lld overflow=%lld\n",
                        (long long)(done - s), (long long)s, ms, 2.0 * nqb * (double)s * h->d / ms / 1e9,
                        m_max, (long long)h->h_gstats[GS_CANDIDATES], overflowed);
            }
            // next slab: expected new hits per query ~ m_max * slab / done; keep the list
            // below ~70 % of its capacity so Poisson noise does not overflow it.
            const double room = 0.01 * h->list_fill_pct * cap - static_cast<double>(m_max);
            double next = room > 0 ? static_cast<double>(done) * room / static_cast<double>(m_max)
                                   : static_cast<double>(TILE_X);
            next = std::min(next, 4.0e9);
            slab = std::max<int64_t>(TILE_X, static_cast<int64_t>(next));
        }

        if (thr_round) {
            exchange_signal_kernel<<<1, 32, 0, h->stream>>>(peer_flags(h->ex), h->ex_seq, XF_THR, h->gstats, 0, dyn);
            h->stats.total_launches++;
        }
        FinalizeParams fp{};
        fp.dyn = dyn;
        fp.dyn_out = h->ex ? 0 : 1;     // exchange: finalize writes the (stable) gather slots
        fp.ring_stages = ring_stages;
        fp.k = k; fp.cap = cap; fp.d = h->d;
        fp.qlist = nullptr;
        fp.cand = cp.cand;
        fp.cnt = reinterpret_cast<int*>(h->kept.p);
        fp.flags = reinterpret_cast<int*>(h->flags.p);
        fp.q32 = qptr; fp.x32 = h->x32;
        fp.x16 = h->x16; fp.d_pad = h->d_pad; fp.sh = h->sh;
        fp.row_offset = h->row_offset;
        fp.n_seg = h->n_seg;
        fp.seg_local = static_cast<const long long*>(h->seg_tab.p);
        fp.seg_delta = fp.seg_local + h->n_seg;
        fp.out_scores = d_scores + q0 * k;
        fp.out_rows = reinterpret_cast<long long*>(d_rows) + q0 * k;
        fp.gstats = h->gstats;
        fp.eps2 = h->two_stage ? reinterpret_cast<const float*>(h->eps2.p) : nullptr;
        fp.cert_eps2 = reinterpret_cast<const float*>(h->eps2.p);
        fp.n_extra = h->n_extra;
        for (int e = 0; e < h->n_extra; e++) {
            fp.extra_r[e] = reinterpret_cast<long long*>(h->extra_base[e]) + q0 * k;
            fp.extra_s[e] = reinterpret_cast<float*>(h->extra_base[e] + static_cast<size_t>(nq) * k * 8) + q0 * k;
            fp.extra_rank[e] = h->extra_rank[e];
        }
        fp.q_base = q0;
        if (h->ex && h->ex->gather_mode == B2IP_GATHER_OWNER) {
            int64_t q_lo, q_hi, per;
            owner_range(h->ex, nq, &q_lo, &q_hi, &per);
            fp.owner_per = static_cast<int>(std::max<int64_t>(per, 1));
            fp.self_rank = h->ex->rank;
        }
        if (thr_round) {
            fp.g_thr = static_cast<const float*>(h->ex->gthr[h->ex->rank]);
            fp.g_flags = static_cast<const unsigned int*>(h->ex->flags[h->ex->rank]);
            fp.g_world = h->ex->world;
            fp.g_stride = h->ex->thr_stride;
            fp.g_seq = h->ex_seq;
            fp.g_timeout_ns = h->ex_timeout_ns;
        }
        if (fuse_refresh) {
            fp.r_cnt = cp.cnt; fp.r_kept = reinterpret_cast<int*>(h->kept.p);
            fp.r_thr = reinterpret_cast<float*>(h->thr.p);
            fp.r_eps2 = reinterpret_cast<const float*>(h->eps2.p);
            fp.r_flags = reinterpret_cast<int*>(h->flags.p);
        }
        cudaEvent_t f0 = get_event(h->ev_fin, 2 * (h->stats.query_batches - 1));
        cudaEvent_t f1 = get_event(h->ev_fin, 2 * (h->stats.query_batches - 1) + 1);
        CAP_TRY(rec(f0));
        // one instantiation per row storage type: the rescore's inner loop is instruction-issue bound
        if (fp.x32) finalize_kernel<true, ROWS_F32><<<nqb, SEL_THREADS, fin_smem, h->stream>>>(fp);
        else if (fp.sh == SH_F16) finalize_kernel<true, ROWS_F16><<<nqb, SEL_THREADS, fin_smem, h->stream>>>(fp);
        else finalize_kernel<true, ROWS_BF16><<<nqb, SEL_THREADS, fin_smem, h->stream>>>(fp);
        CAP_TRY(rec(f1));
        h->stats.total_launches++;
        // end of the device-side search (re-recorded after the exact fallback, if any): the
        // D2H of the counters below and ONE host synchronisation finish the call
        if (q0 + qb >= nq && h->ex) {
            h->ex_prior_overflow = static_cast<long long>(fallback.size());
            CAP_RC(enqueue_exchange(h, nq, k, dyn));
        }
        if (capturing) {
            // the counters' D2H is the graph's last node; instantiate, remember, launch
            CAP_TRY(cudaMemcpyAsync(h->h_gstats, h->gstats, GS_COUNT * sizeof(long long),
                                    cudaMemcpyDeviceToHost, h->stream));
            cudaGraph_t g = nullptr;
            cudaError_t ce = cudaStreamEndCapture(h->stream, &g);
            capturing = false;
            if (ce != cudaSuccess || !g) { cudaGetLastError(); return fail(h, B2IP_ERR_CUDA, "graph capture failed: %s", cudaGetErrorString(ce)); }
            cudaGraphExec_t exec = nullptr;
            ce = cudaGraphInstantiate(&exec, g, 0);
            cudaGraphDestroy(g);
            if (ce != cudaSuccess) { cudaGetLastError(); return fail(h, B2IP_ERR_CUDA, "cudaGraphInstantiate failed: %s", cudaGetErrorString(ce)); }
            if (h->graphs.size() >= 16) {              // drop the least recently used shape
                size_t lru = 0;
                for (size_t i = 1; i < h->graphs.size(); i++)
                    if (h->graphs[i].last_use < h->graphs[lru].last_use) lru = i;
                cudaGraphExecDestroy(h->graphs[lru].exec);
                h->graphs.erase(h->graphs.begin() + static_cast<long>(lru));
            }
            b2ip_index_s::GraphEntry ge{};
            ge.nq = nq; ge.n = n; ge.k = k; ge.cap = cap; ge.ws_gen = h->ws_gen; ge.opt_gen = h->opt_gen;
            ge.has_ex = h->ex != nullptr;
            if (h->ex) ge.ex = *h->ex;
            ge.exec = exec;
            ge.coarse_launches = h->stats.coarse_launches; ge.total_launches = h->stats.total_launches;
            ge.slabs = h->stats.slabs; ge.coarse_flops = h->stats.coarse_flops;
            ge.sample_rows = h->stats.sample_rows;
            ge.ev_used = h->graph_timing ? ev_used : 0;
            ge.last_use = ++h->graph_clock;
            h->graphs.push_back(ge);
            h->graph_captures++;
            h->stats.graph_mode = 1;
            if (!h->graph_timing) ev_used = 0;
            CU_TRY(h, cudaGraphLaunch(exec, h->stream));
        }
        }   // !entry
        if (q0 + qb >= nq) CU_TRY(h, cudaEventRecord(h->ev_t1, h->stream));
        if (!use_graph)
            CU_TRY(h, cudaMemcpyAsync(h->h_gstats, h->gstats, GS_COUNT * sizeof(long long),
                                      cudaMemcpyDeviceToHost, h->stream));
        CU_TRY(h, cudaStreamSynchronize(h->stream));
        CU_TRY(h, cudaGetLastError());
        std::vector<int> hflags;
        if (h->h_gstats[GS_OVERFLOW] > 0) {       // rare: which queries go to the exact path
            hflags.resize(nqb);
            CU_TRY(h, cudaMemcpyAsync(hflags.data(), h->flags.p, nqb * sizeof(int),
                                      cudaMemcpyDeviceToHost, h->stream));
            CU_TRY(h, cudaStreamSynchronize(h->stream));
        }
        h->stats.rescored += h->h_gstats[GS_RESCORED];
        {
            const unsigned int bits = static_cast<unsigned int>(h->h_gstats[GS_MAX_ERR]);
            float r;
            memcpy(&r, &bits, sizeof(r));
            h->stats.max_err_over_eps = std::max(h->stats.max_err_over_eps, static_cast<double>(r));
            h->stats.bound_violations += h->h_gstats[GS_VIOLATIONS];
        }
        h->stats.candidates += h->h_gstats[GS_CANDIDATES];
        for (int i = 0; i < static_cast<int>(hflags.size()); i++)
            if (hflags[i] & FLAG_OVERFLOW) fallback.push_back(static_cast<int>(q0 + i));
    }
#undef CAP_TRY
#undef CAP_RC
    // per-kernel times are read from the recorded event pairs lazily, by b2ip_stats (a dozen
    // cudaEventElapsedTime calls are not free next to a 0.7 ms search)
    h->timing_events = ev_used;
    h->timing_pending = true;
    if (h->verbose) {
        float t = 0.f;
        for (size_t i = 0; i + 3 <= ev_used; i += 3) {
            float a = 0.f, b = 0.f, c = 0.f, gap = 0.f;
            cudaEventElapsedTime(&a, h->ev_t0, h->ev_pool[i]);
            cudaEventElapsedTime(&b, h->ev_pool[i], h->ev_pool[i + 1]);
            cudaEventElapsedTime(&c, h->ev_pool[i + 1], h->ev_pool[i + 2]);
            if (i + 3 < ev_used) cudaEventElapsedTime(&gap, h->ev_pool[i + 2], h->ev_pool[i + 3]);
            fprintf(stderr, "[b2ip] t=%.3f ms: coarse %.3f refresh %.3f then gap %.3f\n", a, b, c, gap);
            t = a + b + c;
        }
        for (int b = 0; b < h->stats.query_batches; b++) {
            float a = 0.f, f = 0.f;
            cudaEventElapsedTime(&a, h->ev_t0, h->ev_fin[2 * b]);
            cudaEventElapsedTime(&f, h->ev_fin[2 * b], h->ev_fin[2 * b + 1]);
            fprintf(stderr, "[b2ip] t=%.3f ms: finalize %.3f (last slab ended at %.3f)\n", a, f, t);
        }
    }
    if (!fallback.empty() && h->ex) {
        // peers have already merged what finalize stored: the caller sees a non-zero exchange
        // status on every rank and repeats the search through the all-gather path
        h->stats.fallback_queries = static_cast<int64_t>(fallback.size());
    } else if (!fallback.empty()) {
        h->stats.fallback_queries = static_cast<int64_t>(fallback.size());
        RC_TRY(exact_search(h, q32, fallback.data(), static_cast<int64_t>(fallback.size()), k,
                            d_scores, d_rows));
        CU_TRY(h, cudaEventRecord(h->ev_t1, h->stream));
        CU_TRY(h, cudaStreamSynchronize(h->stream));
    }
    return B2IP_OK;
}

int search_device(b2ip_handle h, int64_t nq, const float* dq, int k, float* d_scores,
                  int64_t* d_rows, int mode) {
    memset(&h->stats, 0, sizeof(h->stats));
    h->timing_pending = false;
    h->stats.nq = nq; h->stats.ntotal = h->n; h->stats.k = k;
    if (nq == 0) return B2IP_OK;
    CU_TRY(h, cudaEventRecord(h->ev_t0, h->stream));
    if (h->n == 0) {
        fill_padding_kernel<<<256, 256, 0, h->stream>>>(d_scores, reinterpret_cast<long long*>(d_rows), nq * k);
        h->stats.total_launches = 1;
        h->stats.mode_used = B2IP_MODE_EXACT;
        if (h->ex) {      // an empty shard still takes part in the peer-direct exchange
            for (int e = 0; e < h->n_extra; e++)
                fill_padding_kernel<<<256, 256, 0, h->stream>>>(
                    reinterpret_cast<float*>(h->extra_base[e] + static_cast<size_t>(nq) * k * 8),
                    reinterpret_cast<long long*>(h->extra_base[e]), nq * k);
            CU_TRY(h, cudaMemsetAsync(h->gstats, 0, GS_COUNT * sizeof(long long), h->stream));
            h->ex_prior_overflow = 0;
            if (h->ex->gthr[0] && h->ex->thr_stride >= nq) {
                // no rows, no bound: -inf for every query on every rank, then the threshold flag
                for (int r = 0; r < h->ex->world; r++)
                    fill_float_kernel<<<64, 256, 0, h->stream>>>(
                        static_cast<float*>(h->ex->gthr[r]) + static_cast<size_t>(h->ex->rank) * h->ex->thr_stride,
                        nq, -INFINITY);
                exchange_signal_kernel<<<1, 32, 0, h->stream>>>(peer_flags(h->ex), h->ex_seq, XF_THR, h->gstats, 0, nullptr);
            }
            RC_TRY(enqueue_exchange(h, nq, k));
            CU_TRY(h, cudaMemcpyAsync(h->h_gstats, h->gstats, GS_COUNT * sizeof(long long),
                                      cudaMemcpyDeviceToHost, h->stream));
        }
    } else if (mode == B2IP_MODE_EXACT) {
        h->stats.mode_used = B2IP_MODE_EXACT;
        std::vector<int> all(nq);
        for (int64_t i = 0; i < nq; i++) all[i] = static_cast<int>(i);
        RC_TRY(exact_search(h, dq, all.data(), nq, k, d_scores, d_rows));
    } else {
        h->stats.mode_used = B2IP_MODE_TENSOR;
        RC_TRY(tensor_search(h, dq, nq, k, d_scores, d_rows));   // records ev_t1 and synchronises
    }
    if (h->stats.mode_used != B2IP_MODE_TENSOR) {
        CU_TRY(h, cudaEventRecord(h->ev_t1, h->stream));
        CU_TRY(h, cudaStreamSynchronize(h->stream));
    }
    CU_TRY(h, cudaGetLastError());
    if (h->stats.mode_used != B2IP_MODE_TENSOR || h->n == 0) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, h->ev_t0, h->ev_t1);
        h->stats.total_ms = ms;
    }
    return B2IP_OK;
}

}  // namespace

// =========================================================================== C ABI
extern "C" {

const char* b2ip_version(void) { return "b2ip 0.1 sm_100a (tcgen05 bf16 coarse + fp32 rescore)"; }

int b2ip_create(int d, int device, b2ip_handle* out) {
    return b2ip_create_ex(d, device, B2IP_STORE_F32, out);
}

int b2ip_create_ex(int d, int device, int store_dtype, b2ip_handle* out) {
    if (!out) return fail(nullptr, B2IP_ERR_INVALID, "out is NULL");
    *out = nullptr;
    if (store_dtype != B2IP_STORE_F32 && store_dtype != B2IP_STORE_BF16 && store_dtype != B2IP_STORE_F16)
        return fail(nullptr, B2IP_ERR_INVALID, "store_dtype=%d: use B2IP_STORE_F32, B2IP_STORE_F16 or B2IP_STORE_BF16", store_dtype);
    if (d <= 0 || d % 4 != 0 || d > B2IP_MAX_D)
        return fail(nullptr, B2IP_ERR_INVALID, "d=%d: dimension must be a multiple of 4 in [4,%d]", d, B2IP_MAX_D);
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(nullptr, B2IP_ERR_CUDA,
                    "no CUDA device (%s): libb2ip has no CPU fallback", cudaGetErrorString(e));
    }
    if (device < 0 || device >= ndev)
        return fail(nullptr, B2IP_ERR_INVALID, "device %d out of range [0,%d)", device, ndev);
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess)
        return fail(nullptr, B2IP_ERR_CUDA, "cudaGetDeviceProperties(%d) failed", device);
    if (prop.major != 10)
        return fail(nullptr, B2IP_ERR_UNSUPPORTED,
                    "device %d is sm_%d%d; libb2ip is built for sm_100a (B200) only", device,
                    prop.major, prop.minor);
    b2ip_handle h = new b2ip_index_s();
    h->d = d;
    h->store16 = store_dtype != B2IP_STORE_F32;
    h->sh = store_dtype == B2IP_STORE_F16 ? SH_F16 : (store_dtype == B2IP_STORE_BF16 ? SH_BF16 : SH_DEFAULT_F32_STORE);
    if (store_dtype == B2IP_STORE_F32)
        if (const char* s = getenv("B2IP_SHADOW")) h->sh = (s[0] == 'f' || s[0] == 'F') ? SH_F16 : SH_BF16;
    h->d_pad = (d + KBLOCK_ELEMS - 1) / KBLOCK_ELEMS * KBLOCK_ELEMS;
    h->device = device;
    h->sm_count = prop.multiProcessorCount;
    Guard g(device);
    auto bail = [&](int code, const char* what) {
        std::string msg = std::string(what) + ": " + cudaGetErrorString(cudaGetLastError());
        b2ip_destroy(h);
        return fail(nullptr, code, "%s", msg.c_str());
    };
    if (cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking) != cudaSuccess)
        return bail(B2IP_ERR_CUDA, "cudaStreamCreate");
    vmm_init(h);
    h->stream = h->own_stream;
    if (cudaMalloc(&h->norm_stats, 2 * sizeof(unsigned int)) != cudaSuccess ||
        cudaMalloc(&h->gstats, GS_COUNT * sizeof(long long)) != cudaSuccess ||
        cudaMallocHost(&h->h_gstats, GS_COUNT * sizeof(long long)) != cudaSuccess)
        return bail(B2IP_ERR_OOM, "allocating index state");
    if (cudaMalloc(&h->dyn_dev, sizeof(DynArgs)) != cudaSuccess ||
        cudaMallocHost(&h->dyn_host, sizeof(DynArgs)) != cudaSuccess)
        return bail(B2IP_ERR_OOM, "allocating index state");
    if (const char* s = getenv("B2IP_GRAPH")) h->graph = atoi(s);
    if (const char* s = getenv("B2IP_GRAPH_TIMING")) h->graph_timing = atoi(s);
    cudaMemset(h->norm_stats, 0, 2 * sizeof(unsigned int));
    cudaEventCreate(&h->ev_t0);
    cudaEventCreate(&h->ev_t1);
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess || !fn)
        return bail(B2IP_ERR_CUDA, "cuTensorMapEncodeTiled entry point not found");
    h->encode = reinterpret_cast<PFN_encodeTiled>(fn);
    {   // opt-in shared memory sizes, once per process and device
        // (upper bounds for the largest supported d, so handles of different d can coexist)
        const size_t fin_smem = 200u << 10;     // upper bound of finalize_smem_bytes()
        if (cudaFuncSetAttribute(coarse_filter_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, COARSE_SMEM_BYTES) != cudaSuccess ||
            cudaFuncSetAttribute(coarse_filter_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, COARSE_SMEM_BYTES) != cudaSuccess ||
            cudaFuncSetAttribute(coarse_filter_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PAIR_SMEM_BYTES) != cudaSuccess ||
            cudaFuncSetAttribute(coarse_stream_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, MAX_SMEM_OPTIN) != cudaSuccess ||
            cudaFuncSetAttribute(coarse_stream_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, MAX_SMEM_OPTIN) != cudaSuccess ||
            cudaFuncSetAttribute(coarse_stream_kernel<32, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, MAX_SMEM_OPTIN) != cudaSuccess ||
            cudaFuncSetAttribute(coarse_stream_kernel<64, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, MAX_SMEM_OPTIN) != cudaSuccess ||
            cudaFuncSetAttribute(bootstrap_threshold_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, BOOT_MAX_GROUPS * 4) != cudaSuccess ||
            cudaFuncSetAttribute(finalize_kernel<true, ROWS_F32>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(fin_smem)) != cudaSuccess ||
            cudaFuncSetAttribute(finalize_kernel<true, ROWS_BF16>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(fin_smem)) != cudaSuccess ||
            cudaFuncSetAttribute(finalize_kernel<true, ROWS_F16>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(fin_smem)) != cudaSuccess ||
            cudaFuncSetAttribute(finalize_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(fin_smem)) != cudaSuccess ||
            cudaFuncSetAttribute(exact_scores_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 static_cast<int>(static_cast<size_t>(EXACT_QB) * B2IP_MAX_D * sizeof(float))) != cudaSuccess)
            return bail(B2IP_ERR_CUDA, "cudaFuncSetAttribute(MaxDynamicSharedMemorySize)");
    }
    h->gx = std::max(1, h->sm_count / 2);   // = clusters of the pair kernel: one query tile per wave,
                                            // the corpus tiles of a group stay L2 resident (measured best)
    if (const char* s = getenv("B2IP_GX")) h->gx = std::max(1, atoi(s));
    if (const char* s = getenv("B2IP_STREAM_KERNEL")) h->stream_kernel = atoi(s);
    if (const char* s = getenv("B2IP_BOOTSTRAP")) h->bootstrap = atoi(s);
    if (const char* s = getenv("B2IP_BOOTSTRAP_MAX_MB")) h->bootstrap_max_mb = std::max(0, atoi(s));
    if (const char* s = getenv("B2IP_HINT_Q")) h->hint_q = atoi(s);
    if (const char* s = getenv("B2IP_HINT_X")) h->hint_x = atoi(s);
    if (const char* s = getenv("B2IP_CAND_BUDGET_MB")) h->cand_budget_bytes = std::max(1ll, atoll(s)) << 20;
    if (const char* s = getenv("B2IP_EXCHANGE_TIMEOUT_S"))
        h->ex_timeout_ns = static_cast<long long>(std::max(0.001, atof(s)) * 1e9);
    memset(&h->stats, 0, sizeof(h->stats));
    *out = h;
    return B2IP_OK;
}

void b2ip_destroy(b2ip_handle h) {
    if (!h) return;
    Guard g(h->device);
    if (h->own_stream) cudaStreamSynchronize(h->own_stream);
    for (DevBuf* b : {&h->q16, &h->eps2, &h->thr, &h->cnt, &h->kept, &h->flags, &h->cand, &h->qstage, &h->qhalf,
                      &h->out_s, &h->out_r, &h->exact_scores, &h->exact_misc, &h->qlist, &h->stage,
                      &h->seg_tab, &h->gmax})
        release(*b);
    if (h->v16.base || h->v32.base) {
        vmm_free(h, h->v32);
        vmm_free(h, h->v16);
    } else {
        if (h->x32) cudaFree(h->x32);
        if (h->x16) cudaFree(h->x16);
    }
    if (h->norm_stats) cudaFree(h->norm_stats);
    if (h->gstats) cudaFree(h->gstats);
    if (h->h_gstats) cudaFreeHost(h->h_gstats);
    for (auto& ge : h->graphs) cudaGraphExecDestroy(ge.exec);
    if (h->dyn_dev) cudaFree(h->dyn_dev);
    if (h->dyn_host) cudaFreeHost(h->dyn_host);
    delete h->pool;
    for (int b = 0; b < 2; b++) {
        if (h->pin[b]) cudaFreeHost(h->pin[b]);
        if (h->pin_ev[b]) cudaEventDestroy(h->pin_ev[b]);
    }
    for (cudaEvent_t e : h->ev_pool) cudaEventDestroy(e);
    for (cudaEvent_t e : h->ev_fin) cudaEventDestroy(e);
    if (h->ev_t0) cudaEventDestroy(h->ev_t0);
    if (h->ev_t1) cudaEventDestroy(h->ev_t1);
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    delete h;
}

int b2ip_set_stream(b2ip_handle h, void* cuda_stream) {
    if (!h) return B2IP_ERR_INVALID;
    h->stream = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : h->own_stream;
    h->opt_gen++;
    return B2IP_OK;
}

int b2ip_set_option(b2ip_handle h, const char* name, int64_t value) {
    if (!h || !name) return B2IP_ERR_INVALID;
    const std::string n(name);
    h->opt_gen++;
    if (n == "gx") h->gx = static_cast<int>(std::max<int64_t>(1, value));
    else if (n == "hint_q") h->hint_q = static_cast<int>(value);
    else if (n == "hint_x") h->hint_x = static_cast<int>(value);
    else if (n == "dbg") {
        // perf experiments that BREAK results (see CoarseParams::dbg): only with B2IP_DEBUG=1
        const char* e = getenv("B2IP_DEBUG");
        if (!e || atoi(e) == 0) return fail(h, B2IP_ERR_INVALID, "option 'dbg' needs B2IP_DEBUG=1 in the environment");
        h->dbg = static_cast<int>(value);
    }
    else if (n == "verbose") h->verbose = static_cast<int>(value);
    else if (n == "pair") h->pair = static_cast<int>(value);
    else if (n == "dense_first") h->dense_first = static_cast<int>(value);
    else if (n == "bootstrap") h->bootstrap = static_cast<int>(value);
    else if (n == "bootstrap_max_mb") h->bootstrap_max_mb = static_cast<int>(std::min<int64_t>(std::max<int64_t>(0, value), 1 << 20));
    else if (n == "stream_kernel") h->stream_kernel = static_cast<int>(value);
    else if (n == "list_fill_pct") h->list_fill_pct = std::min(90, std::max(10, static_cast<int>(value)));
    else if (n == "fuse_refresh") h->fuse_refresh = static_cast<int>(value);
    else if (n == "two_stage") h->two_stage = static_cast<int>(value);
    else if (n == "cand_budget_mb") h->cand_budget_bytes = std::max<int64_t>(1, value) << 20;
    else if (n == "graph") h->graph = static_cast<int>(value);
    else if (n == "graph_timing") h->graph_timing = static_cast<int>(value);
    else if (n == "shadow_f16") {
        // operand type of the coarse pass of an fp32-stored index; only before the first row
        if (h->store16) return fail(h, B2IP_ERR_INVALID, "shadow_f16: a 16-bit store fixes the operand type");
        if (h->n > 0) return fail(h, B2IP_ERR_INVALID, "shadow_f16: set before the first b2ip_add");
        h->sh = value ? SH_F16 : SH_BF16;
    }
    else return fail(h, B2IP_ERR_INVALID, "b2ip_set_option: unknown option '%s'", name);
    return B2IP_OK;
}

int b2ip_reserve(b2ip_handle h, int64_t n_rows) {
    if (!h) return B2IP_ERR_INVALID;
    if (n_rows < 0 || n_rows >= (1ll << 31) - 512) return fail(h, B2IP_ERR_INVALID, "n_rows=%lld out of range", (long long)n_rows);
    Guard g(h->device);
    if (n_rows <= h->cap_rows) return B2IP_OK;
    return grow_rows(h, n_rows, /*exact=*/true);   // a reserve states the final size
}

int b2ip_add(b2ip_handle h, int64_t n, const void* rows, int src_dtype, int mem) {
    if (!h) return B2IP_ERR_INVALID;
    if (n < 0 || (n > 0 && !rows)) return fail(h, B2IP_ERR_INVALID, "b2ip_add: bad rows pointer / n=%lld", (long long)n);
    if (src_dtype != B2IP_F32 && src_dtype != B2IP_F16 && src_dtype != B2IP_BF16)
        return fail(h, B2IP_ERR_INVALID, "b2ip_add: src_dtype=%d", src_dtype);
    if (mem != B2IP_MEM_HOST && mem != B2IP_MEM_DEVICE) return fail(h, B2IP_ERR_INVALID, "b2ip_add: mem=%d", mem);
    if (src_dtype == B2IP_BF16 && !(h->store16 && h->sh == SH_BF16))
        return fail(h, B2IP_ERR_INVALID, "b2ip_add: bf16 rows need an index created with B2IP_STORE_BF16");
    // rows handed in in the storage type itself are copied as they are
    const bool same16 = h->store16 && ((src_dtype == B2IP_BF16 && h->sh == SH_BF16) ||
                                       (src_dtype == B2IP_F16 && h->sh == SH_F16));
    if (n == 0) return B2IP_OK;
    if (h->n + n >= (1ll << 31) - 512) return fail(h, B2IP_ERR_UNSUPPORTED, "a shard holds at most 2^31-512 rows (TMA coordinates are int32)");
    Guard g(h->device);
    RC_TRY(grow_rows(h, h->n + n));
    const bool host = mem == B2IP_MEM_HOST;
    const size_t elem = src_dtype == B2IP_F32 ? 4 : 2;
    const size_t row_bytes = static_cast<size_t>(h->d) * elem;
    // Rows are processed in chunks: each chunk is landed on the device (host rows go through
    // the double-buffered pinned staging of host_to_device, so the CPU-side copy of chunk i+1
    // overlaps the DMA and the conversion kernels of chunk i), converted, and shadowed.
    const bool lands_in_master = host && src_dtype == B2IP_F32 && !h->store16;
    const bool need_f32_stage = h->store16 && !same16 && !(src_dtype == B2IP_F32 && !host);
    // device rows that need no staging area are converted in one piece
    const int64_t chunk = (!host && !need_f32_stage)
        ? n : std::max<int64_t>(1, std::min<int64_t>(n, INGEST_CHUNK_BYTES / static_cast<int64_t>(row_bytes)));
    const size_t land_bytes = (host && !lands_in_master) ? static_cast<size_t>(chunk) * row_bytes : 0;
    const size_t land_pad = (land_bytes + 255) & ~static_cast<size_t>(255);
    if (land_bytes || need_f32_stage)
        RC_TRY(ensure(h, h->stage, land_pad + (need_f32_stage ? static_cast<size_t>(chunk) * h->d * sizeof(float) : 0)));
    for (int64_t c0 = 0; c0 < n; c0 += chunk) {
        const int64_t cn = std::min<int64_t>(chunk, n - c0);
        const size_t count = static_cast<size_t>(cn) * h->d;
        const int64_t r0 = h->n + c0;
        const int rgrid = static_cast<int>(std::min<int64_t>((cn + 7) / 8, static_cast<int64_t>(h->sm_count) * 16));
        const char* src_any = static_cast<const char*>(rows) + static_cast<size_t>(c0) * row_bytes;
        float* master = h->store16 ? nullptr : h->x32 + r0 * h->d;
        const void* src_dev = src_any;                       // this chunk's source rows, on the device
        if (host) {
            void* land = lands_in_master ? static_cast<void*>(master) : h->stage.p;
            RC_TRY(host_to_device(h, land, src_any, count * elem));
            src_dev = land;
        }
        if (same16) {
            ingest_16bit_rows_kernel<<<rgrid, 256, 0, h->stream>>>(
                static_cast<const __nv_bfloat16*>(src_dev), h->x16, r0, r0 + cn, h->d, h->d_pad,
                h->norm_stats, h->sh);
            continue;
        }
        // fp32 view of the chunk: the master rows, the caller's device buffer, or the staging area
        const float* p32;
        if (src_dtype == B2IP_F32) {
            p32 = static_cast<const float*>(src_dev);
            if (master && p32 != master) {
                CU_TRY(h, cudaMemcpyAsync(master, p32, count * sizeof(float), cudaMemcpyDeviceToDevice, h->stream));
                p32 = master;
            }
        } else {
            float* dst32 = master ? master : reinterpret_cast<float*>(static_cast<char*>(h->stage.p) + land_pad);
            const int grid = static_cast<int>(std::min<size_t>((count / 2 + 255) / 256 + 1, 65535));
            widen_f16_kernel<<<grid, 256, 0, h->stream>>>(static_cast<const __half*>(src_dev), dst32,
                                                         static_cast<long long>(count));
            p32 = dst32;
        }
        shadow_rows_kernel<<<rgrid, 256, 0, h->stream>>>(p32, r0, h->x16, r0, r0 + cn, h->d, h->d_pad,
                                                         h->norm_stats, !h->store16, h->sh);
    }
    CU_TRY(h, cudaGetLastError());
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    h->n += n;
    return B2IP_OK;
}

int64_t b2ip_ntotal(b2ip_handle h) { return h ? h->n : -1; }
int b2ip_dim(b2ip_handle h) { return h ? h->d : -1; }

// Global row ids travel through the merge kernels as 32-bit key halves (keys.cuh): a sharded
// index may hold at most 2^32 - 1 rows in total.  Checked where ids are assigned and at search time.
constexpr int64_t MAX_GLOBAL_ROWS = 0xFFFFFFFFll;

int b2ip_set_row_offset(b2ip_handle h, int64_t offset) {
    if (!h || offset < 0) return B2IP_ERR_INVALID;
    if (offset + h->n > MAX_GLOBAL_ROWS)
        return fail(h, B2IP_ERR_UNSUPPORTED, "b2ip_set_row_offset: offset %lld + %lld rows exceeds the 2^32 - 1 global row ids "
                    "the merge supports", (long long)offset, (long long)h->n);
    h->opt_gen++;
    h->row_offset = offset;
    return B2IP_OK;
}

int b2ip_set_row_segments(b2ip_handle h, int n_segments, const int64_t* local_start,
                          const int64_t* global_start) {
    if (!h || n_segments < 0 || (n_segments > 0 && (!local_start || !global_start)))
        return fail(h, B2IP_ERR_INVALID, "b2ip_set_row_segments: bad arguments");
    for (int i = 0; i < n_segments; i++) {
        if (local_start[i] < 0 || global_start[i] < 0 || (i == 0 && local_start[0] != 0) ||
            (i > 0 && (local_start[i] <= local_start[i - 1] || global_start[i] <= global_start[i - 1])))
            return fail(h, B2IP_ERR_INVALID, "b2ip_set_row_segments: segment %d out of order", i);
    }
    if (n_segments > 0) {
        // the last segment reaches the highest id: global_start + (rows held - its local start)
        const int64_t top = global_start[n_segments - 1] + std::max<int64_t>(h->n - local_start[n_segments - 1], 0);
        if (top > MAX_GLOBAL_ROWS)
            return fail(h, B2IP_ERR_UNSUPPORTED, "b2ip_set_row_segments: global row ids up to %lld exceed 2^32 - 1", (long long)top);
    }
    Guard g(h->device);
    if (n_segments > 0) {
        std::vector<long long> tab(2 * static_cast<size_t>(n_segments));
        for (int i = 0; i < n_segments; i++) {
            tab[i] = local_start[i];
            tab[n_segments + i] = global_start[i] - local_start[i];
        }
        CU_TRY(h, cudaStreamSynchronize(h->stream));
        RC_TRY(ensure(h, h->seg_tab, tab.size() * sizeof(long long)));
        CU_TRY(h, cudaMemcpyAsync(h->seg_tab.p, tab.data(), tab.size() * sizeof(long long),
                                  cudaMemcpyHostToDevice, h->stream));
        CU_TRY(h, cudaStreamSynchronize(h->stream));
    }
    h->n_seg = n_segments;
    h->opt_gen++;
    return B2IP_OK;
}

int b2ip_search(b2ip_handle h, int64_t nq, const float* queries, int k, float* out_scores,
                int64_t* out_rows, int mode, int mem) {
    return b2ip_search_ex(h, nq, queries, B2IP_F32, k, out_scores, out_rows, mode, mem);
}

int b2ip_search_ex(b2ip_handle h, int64_t nq, const void* queries_any, int q_dtype, int k,
                   float* out_scores, int64_t* out_rows, int mode, int mem) {
    if (!h) return B2IP_ERR_INVALID;
    if (q_dtype != B2IP_F32 && q_dtype != B2IP_F16)
        return fail(h, B2IP_ERR_INVALID, "b2ip_search: q_dtype=%d (use B2IP_F32 or B2IP_F16)", q_dtype);
    const float* queries = static_cast<const float*>(queries_any);
    if (nq < 0 || (nq > 0 && (!queries || !out_scores || !out_rows)))
        return fail(h, B2IP_ERR_INVALID, "b2ip_search: NULL buffer or nq=%lld", (long long)nq);
    if (k < 1) return fail(h, B2IP_ERR_INVALID, "b2ip_search: k=%d must be >= 1", k);
    if (k > B2IP_MAX_K) return fail(h, B2IP_ERR_UNSUPPORTED, "b2ip_search: k=%d above B2IP_MAX_K=%d", k, B2IP_MAX_K);
    if (mode < B2IP_MODE_AUTO || mode > B2IP_MODE_EXACT) return fail(h, B2IP_ERR_INVALID, "b2ip_search: mode=%d", mode);
    if (mem != B2IP_MEM_HOST && mem != B2IP_MEM_DEVICE) return fail(h, B2IP_ERR_INVALID, "b2ip_search: mem=%d", mem);
    if (nq >= (1ll << 31)) return fail(h, B2IP_ERR_UNSUPPORTED, "b2ip_search: nq too large");
    if (h->n_seg == 0 && h->row_offset + h->n > MAX_GLOBAL_ROWS)
        return fail(h, B2IP_ERR_UNSUPPORTED, "b2ip_search: row offset %lld + %lld rows exceeds 2^32 - 1 global row ids",
                    (long long)h->row_offset, (long long)h->n);
    Guard g(h->device);
    if (nq == 0) { memset(&h->stats, 0, sizeof(h->stats)); h->timing_pending = false; return B2IP_OK; }
    const size_t q_count = static_cast<size_t>(nq) * h->d;
    // float16 queries are widened on the GPU: exactly what `query_vectors.astype('float32')`
    // (src/index.py:35) does on the host, without the host pass and with half the H2D bytes
    auto widen_queries = [&](const void* half_dev) {
        const int grid = static_cast<int>(std::min<size_t>((q_count / 2 + 255) / 256 + 1, 65535));
        widen_f16_kernel<<<grid, 256, 0, h->stream>>>(static_cast<const __half*>(half_dev),
                                                      static_cast<float*>(h->qstage.p),
                                                      static_cast<long long>(q_count));
    };
    if (mem == B2IP_MEM_DEVICE) {
        if (q_dtype == B2IP_F32) return search_device(h, nq, queries, k, out_scores, out_rows, mode);
        RC_TRY(ensure(h, h->qstage, q_count * sizeof(float)));
        widen_queries(queries_any);
        return search_device(h, nq, static_cast<const float*>(h->qstage.p), k, out_scores, out_rows, mode);
    }
    RC_TRY(ensure(h, h->qstage, q_count * sizeof(float)));
    RC_TRY(ensure(h, h->out_s, static_cast<size_t>(nq) * k * sizeof(float)));
    RC_TRY(ensure(h, h->out_r, static_cast<size_t>(nq) * k * sizeof(int64_t)));
    if (q_dtype == B2IP_F16) {
        RC_TRY(ensure(h, h->qhalf, q_count * 2));
        RC_TRY(host_to_device(h, h->qhalf.p, queries_any, q_count * 2));
        widen_queries(h->qhalf.p);
    } else {
        RC_TRY(host_to_device(h, h->qstage.p, queries, q_count * sizeof(float)));
    }
    RC_TRY(search_device(h, nq, static_cast<const float*>(h->qstage.p), k,
                         static_cast<float*>(h->out_s.p), static_cast<int64_t*>(h->out_r.p), mode));
    const size_t sb = static_cast<size_t>(nq) * k * sizeof(float), rb = static_cast<size_t>(nq) * k * sizeof(int64_t);
    cudaPointerAttributes a1, a2;
    const bool pin1 = cudaPointerGetAttributes(&a1, out_scores) == cudaSuccess && a1.type != cudaMemoryTypeUnregistered;
    const bool pin2 = cudaPointerGetAttributes(&a2, out_rows) == cudaSuccess && a2.type != cudaMemoryTypeUnregistered;
    cudaGetLastError();
    if ((pin1 && pin2) || sb + rb < (512u << 10)) {      // both on the copy engine, one synchronisation
        CU_TRY(h, cudaMemcpyAsync(out_scores, h->out_s.p, sb, cudaMemcpyDeviceToHost, h->stream));
        CU_TRY(h, cudaMemcpyAsync(out_rows, h->out_r.p, rb, cudaMemcpyDeviceToHost, h->stream));
        CU_TRY(h, cudaStreamSynchronize(h->stream));
        return B2IP_OK;
    }
    RC_TRY(device_to_host(h, out_scores, h->out_s.p, sb));
    RC_TRY(device_to_host(h, out_rows, h->out_r.p, rb));
    return B2IP_OK;
}

int b2ip_search_exchange(b2ip_handle h, int64_t nq, const float* queries_dev, int k,
                         const b2ip_exchange_t* ex, uint32_t seq, float* out_scores_dev,
                         int64_t* out_rows_dev, int64_t* status) {
    if (!h) return B2IP_ERR_INVALID;
    if (!ex || !status || nq <= 0 || !queries_dev)
        return fail(h, B2IP_ERR_INVALID, "b2ip_search_exchange: NULL argument or nq=%lld", (long long)nq);
    if (k < 1 || k > B2IP_MAX_K) return fail(h, B2IP_ERR_UNSUPPORTED, "b2ip_search_exchange: k=%d", k);
    if (ex->world < 1 || ex->world > B2IP_MAX_PEERS || ex->rank < 0 || ex->rank >= ex->world)
        return fail(h, B2IP_ERR_INVALID, "b2ip_search_exchange: world=%d rank=%d", ex->world, ex->rank);
    if (ex->slot_bytes % 16 != 0 || ex->slot_bytes < nq * k * 12)
        return fail(h, B2IP_ERR_INVALID, "b2ip_search_exchange: slot_bytes=%lld for nq*k=%lld", (long long)ex->slot_bytes, (long long)(nq * k));
    Guard g(h->device);
    // this rank's block goes to slot `rank` of every rank's gather buffer; the local one is the
    // primary output of the finalize kernel, the others its extra (peer) outputs
    char* mine = static_cast<char*>(ex->gather[ex->rank]) + static_cast<size_t>(ex->rank) * ex->slot_bytes;
    if (ex->gather_mode != B2IP_GATHER_ALL && ex->gather_mode != B2IP_GATHER_OWNER)
        return fail(h, B2IP_ERR_INVALID, "b2ip_search_exchange: gather_mode=%d", ex->gather_mode);
    {   // the output buffers may be NULL only when this rank owns no query of the search
        int64_t q_lo = 0, q_hi = nq, per = 0;
        if (ex->gather_mode == B2IP_GATHER_OWNER) owner_range(ex, nq, &q_lo, &q_hi, &per);
        if (q_hi > q_lo && (!out_scores_dev || !out_rows_dev))
            return fail(h, B2IP_ERR_INVALID, "b2ip_search_exchange: NULL output buffer");
    }
    h->n_extra = 0;
    for (int p = 0; p < ex->world; p++)
        if (p != ex->rank) {
            h->extra_rank[h->n_extra] = p;
            h->extra_base[h->n_extra++] = static_cast<char*>(ex->gather[p]) + static_cast<size_t>(ex->rank) * ex->slot_bytes;
        }
    h->ex = ex;
    h->ex_seq = seq;
    h->ex_out_s = out_scores_dev;
    h->ex_out_r = out_rows_dev;
    const int rc = search_device(h, nq, queries_dev, k, reinterpret_cast<float*>(mine + static_cast<size_t>(nq) * k * 8),
                                 reinterpret_cast<int64_t*>(mine), B2IP_MODE_TENSOR);
    h->ex = nullptr;
    h->n_extra = 0;
    if (rc != B2IP_OK) return rc;
    *status = h->h_gstats[GS_XSTATUS];
    if (*status >= XSTATUS_TIMEOUT)
        return fail(h, B2IP_ERR_INTERNAL,
                    "b2ip_search_exchange: a peer's flag for search %u did not arrive within %.0f s "
                    "(B2IP_EXCHANGE_TIMEOUT_S): the peer is gone or stuck; this rank's view of the "
                    "exchange is no longer consistent with its peers -- tear the process group down",
                    seq, h->ex_timeout_ns * 1e-9);
    return B2IP_OK;
}

namespace {
constexpr size_t GROUP_FLAG_BYTES = 256;

void group_run(b2ip_group g, std::function<void(int)> f) {
    std::unique_lock<std::mutex> l(g->m);
    g->job = std::move(f);
    g->left = static_cast<int>(g->hs.size());
    g->gen++;
    g->cv.notify_all();
    g->done.wait(l, [g] { return g->left == 0; });
}

void group_worker(b2ip_group g, int i) {
    unsigned long long seen = 0;
    std::unique_lock<std::mutex> l(g->m);
    for (;;) {
        g->cv.wait(l, [&] { return g->gen != seen || g->stop; });
        if (g->stop) return;
        seen = g->gen;
        std::function<void(int)> f = g->job;
        l.unlock();
        f(i);
        l.lock();
        if (--g->left == 0) g->done.notify_one();
    }
}

void group_free_buffers(b2ip_group g) {
    for (size_t i = 0; i < g->buf.size(); i++)
        if (g->buf[i]) { Guard gd(g->hs[i]->device); cudaFree(g->buf[i]); g->buf[i] = nullptr; }
}

// (re)allocates the exchange buffers for searches of up to nq queries and k results
int group_buffers(b2ip_group g, int64_t nq, int k) {
    const size_t need = (static_cast<size_t>(nq) * k * 12 + 15) / 16 * 16;
    if (!g->buf.empty() && g->buf[0] && need <= g->slot && static_cast<size_t>(nq) <= g->thr_cap) return B2IP_OK;
    const int G = static_cast<int>(g->hs.size());
    const size_t slot = std::max<size_t>(std::max<size_t>(1 << 16, (need + need / 4 + 65535) / 65536 * 65536), g->slot);
    const size_t thr_cap = std::max<size_t>((static_cast<size_t>(nq) + nq / 4 + 1023) / 1024 * 1024, g->thr_cap);
    const size_t thr_bytes = static_cast<size_t>(G) * thr_cap * 4;
    const size_t total = 2 * G * slot + 2 * thr_bytes + 2 * GROUP_FLAG_BYTES;
    for (int i = 0; i < G; i++) { Guard gd(g->hs[i]->device); cudaStreamSynchronize(g->hs[i]->stream); }
    group_free_buffers(g);
    g->buf.assign(G, nullptr);
    for (int i = 0; i < G; i++) {
        Guard gd(g->hs[i]->device);
        void* p = nullptr;
        cudaError_t e = cudaMalloc(&p, total);
        if (e == cudaSuccess) e = cudaMemset(p, 0, total);
        if (e == cudaSuccess) e = cudaDeviceSynchronize();
        if (e != cudaSuccess) {
            cudaGetLastError();
            g->err = std::string("group exchange buffers: ") + cudaGetErrorString(e);
            group_free_buffers(g);
            return e == cudaErrorMemoryAllocation ? B2IP_ERR_OOM : B2IP_ERR_CUDA;
        }
        g->buf[i] = static_cast<char*>(p);
    }
    for (int parity = 0; parity < 2; parity++)
        for (int i = 0; i < G; i++) {
            b2ip_exchange_t& ex = g->ex[parity][i];
            memset(&ex, 0, sizeof(ex));
            ex.world = G; ex.rank = i; ex.slot_bytes = static_cast<int64_t>(slot);
            ex.thr_stride = static_cast<int64_t>(thr_cap);
            ex.gather_mode = B2IP_GATHER_OWNER;
            for (int p = 0; p < G; p++) {
                ex.gather[p] = g->buf[p] + parity * G * slot;
                ex.gthr[p] = g->buf[p] + 2 * G * slot + parity * thr_bytes;
                ex.flags[p] = g->buf[p] + 2 * G * slot + 2 * thr_bytes + parity * GROUP_FLAG_BYTES;
            }
        }
    g->slot = slot; g->thr_cap = thr_cap; g->seq = 0;
    return B2IP_OK;
}
}  // namespace

int b2ip_group_create(int n_handles, const b2ip_handle* handles, b2ip_group* out) {
    if (!out) return B2IP_ERR_INVALID;
    *out = nullptr;
    if (n_handles < 1 || n_handles > B2IP_MAX_PEERS || !handles)
        return fail(nullptr, B2IP_ERR_INVALID, "b2ip_group_create: n_handles=%d (1..%d)", n_handles, B2IP_MAX_PEERS);
    for (int i = 0; i < n_handles; i++) {
        if (!handles[i]) return fail(nullptr, B2IP_ERR_INVALID, "b2ip_group_create: NULL handle");
        if (handles[i]->d != handles[0]->d) return fail(nullptr, B2IP_ERR_INVALID, "b2ip_group_create: handles differ in d");
        for (int j = 0; j < i; j++)
            if (handles[j]->device == handles[i]->device)
                return fail(nullptr, B2IP_ERR_INVALID, "b2ip_group_create: two handles on device %d", handles[i]->device);
    }
    // every member's kernels store into every other member's buffers
    for (int i = 0; i < n_handles; i++)
        for (int j = 0; j < n_handles; j++) {
            const int rc = b2ip_enable_peer_access(handles[i], handles[j]->device);
            if (rc != B2IP_OK) return fail(nullptr, rc, "b2ip_group_create: %s", handles[i]->err.c_str());
        }
    b2ip_group g = new b2ip_group_s();
    g->hs.assign(handles, handles + n_handles);
    for (int i = 0; i < n_handles; i++) g->th.emplace_back(group_worker, g, i);
    *out = g;
    return B2IP_OK;
}

void b2ip_group_destroy(b2ip_group g) {
    if (!g) return;
    { std::lock_guard<std::mutex> l(g->m); g->stop = true; }
    g->cv.notify_all();
    for (auto& t : g->th) t.join();
    group_free_buffers(g);
    delete g;
}

const char* b2ip_group_last_error(b2ip_group g) { return g ? g->err.c_str() : g_create_error.c_str(); }

int b2ip_group_search(b2ip_group g, int64_t nq, const void* queries_host, int q_dtype, int k,
                      float* out_scores_host, int64_t* out_rows_host, int64_t* status) {
    if (!g || !status) return B2IP_ERR_INVALID;
    *status = 0;
    if (q_dtype != B2IP_F32 && q_dtype != B2IP_F16) { g->err = "b2ip_group_search: q_dtype"; return B2IP_ERR_INVALID; }
    if (nq < 0 || (nq > 0 && (!queries_host || !out_scores_host || !out_rows_host)) || k < 1 || k > B2IP_MAX_K) {
        g->err = "b2ip_group_search: bad arguments";
        return B2IP_ERR_INVALID;
    }
    if (nq == 0) return B2IP_OK;
    const int rcb = group_buffers(g, nq, k);
    if (rcb != B2IP_OK) return rcb;
    const int G = static_cast<int>(g->hs.size());
    const unsigned int seq = ++g->seq;
    const int parity = static_cast<int>(seq & 1);
    const int64_t per = (nq + G - 1) / G;
    std::vector<int> rcs(G, B2IP_OK);
    std::vector<int64_t> sts(G, 0);
    group_run(g, [&](int i) {
        b2ip_handle h = g->hs[i];
        Guard gd(h->device);
        auto run = [&]() -> int {
            const size_t q_count = static_cast<size_t>(nq) * h->d;
            const int64_t q_lo = std::min<int64_t>(i * per, nq), q_hi = std::min<int64_t>(q_lo + per, nq);
            RC_TRY(ensure(h, h->qstage, q_count * sizeof(float)));
            RC_TRY(ensure(h, h->out_s, static_cast<size_t>(per) * k * sizeof(float)));
            RC_TRY(ensure(h, h->out_r, static_cast<size_t>(per) * k * sizeof(int64_t)));
            // every member uploads the queries itself: G host->device copies run in parallel on G links
            if (q_dtype == B2IP_F16) {
                RC_TRY(ensure(h, h->qhalf, q_count * 2));
                RC_TRY(host_to_device(h, h->qhalf.p, queries_host, q_count * 2));
                const int grid = static_cast<int>(std::min<size_t>((q_count / 2 + 255) / 256 + 1, 65535));
                widen_f16_kernel<<<grid, 256, 0, h->stream>>>(static_cast<const __half*>(h->qhalf.p),
                                                              static_cast<float*>(h->qstage.p),
                                                              static_cast<long long>(q_count));
            } else {
                RC_TRY(host_to_device(h, h->qstage.p, queries_host, q_count * sizeof(float)));
            }
            RC_TRY(b2ip_search_exchange(h, nq, static_cast<const float*>(h->qstage.p), k, &g->ex[parity][i], seq,
                                        static_cast<float*>(h->out_s.p), static_cast<int64_t*>(h->out_r.p), &sts[i]));
            if (sts[i] == 0 && q_hi > q_lo) {
                // this member's slice of the answer leaves on its own copy engine
                RC_TRY(device_to_host(h, out_scores_host + q_lo * k, h->out_s.p, static_cast<size_t>(q_hi - q_lo) * k * sizeof(float)));
                RC_TRY(device_to_host(h, out_rows_host + q_lo * k, h->out_r.p, static_cast<size_t>(q_hi - q_lo) * k * sizeof(int64_t)));
            }
            return B2IP_OK;
        };
        rcs[i] = run();
    });
    for (int i = 0; i < G; i++) {
        if (rcs[i] != B2IP_OK) {
            g->err = "member " + std::to_string(i) + ": " + g->hs[i]->err;
            return rcs[i];
        }
        *status = std::max(*status, sts[i]);
    }
    return B2IP_OK;
}

int b2ip_enable_peer_access(b2ip_handle h, int peer_device) {
    if (!h) return B2IP_ERR_INVALID;
    if (peer_device == h->device) return B2IP_OK;
    Guard g(h->device);
    int can = 0;
    CU_TRY(h, cudaDeviceCanAccessPeer(&can, h->device, peer_device));
    if (!can) return fail(h, B2IP_ERR_UNSUPPORTED, "device %d cannot access device %d (no P2P path)", h->device, peer_device);
    cudaError_t e = cudaDeviceEnablePeerAccess(peer_device, 0);
    if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); return B2IP_OK; }
    CU_TRY(h, e);
    return B2IP_OK;
}

int b2ip_merge_topk(int device, void* cuda_stream, int64_t nq, int k, int n_lists,
                    const float* scores, const int64_t* rows, float* out_scores, int64_t* out_rows) {
    return b2ip_merge_topk_strided(device, cuda_stream, nq, k, n_lists, scores, rows, nq * k, nq * k,
                                   out_scores, out_rows);
}

int b2ip_merge_topk_strided(int device, void* cuda_stream, int64_t nq, int k, int n_lists,
                            const float* scores, const int64_t* rows, int64_t scores_list_stride,
                            int64_t rows_list_stride, float* out_scores, int64_t* out_rows) {
    if (nq < 0 || k < 1 || k > B2IP_MAX_K || n_lists < 1 || n_lists > 64)
        return fail(nullptr, B2IP_ERR_INVALID, "b2ip_merge_topk: nq=%lld k=%d n_lists=%d", (long long)nq, k, n_lists);
    if (nq == 0) return B2IP_OK;
    if (!scores || !rows || !out_scores || !out_rows) return fail(nullptr, B2IP_ERR_INVALID, "b2ip_merge_topk: NULL buffer");
    Guard g(device);
    int P = 2;
    while (P < n_lists * k) P <<= 1;
    const size_t smem = static_cast<size_t>(P) * sizeof(unsigned long long);
    if (smem > 200 * 1024) return fail(nullptr, B2IP_ERR_UNSUPPORTED, "b2ip_merge_topk: n_lists*k=%d too large", n_lists * k);
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    cudaError_t e = cudaFuncSetAttribute(merge_topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e == cudaSuccess) {
        merge_topk_kernel<<<static_cast<unsigned int>(nq), SEL_THREADS, smem, st>>>(
            nq, k, n_lists, scores, reinterpret_cast<const long long*>(rows), scores_list_stride,
            rows_list_stride, out_scores, reinterpret_cast<long long*>(out_rows), P, nullptr, 0u, nullptr, 0, 0, nullptr);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(nullptr, B2IP_ERR_CUDA, "b2ip_merge_topk: %s", cudaGetErrorString(e)); }
    return B2IP_OK;
}

int b2ip_export_rows(b2ip_handle h, int64_t row0, int64_t n, float* out, int mem) {
    if (!h) return B2IP_ERR_INVALID;
    if (row0 < 0 || n < 0 || row0 + n > h->n || (n > 0 && !out))
        return fail(h, B2IP_ERR_INVALID, "b2ip_export_rows: [%lld,+%lld) outside [0,%lld)", (long long)row0, (long long)n, (long long)h->n);
    if (n == 0) return B2IP_OK;
    Guard g(h->device);
    const float* src = h->x32 ? h->x32 + row0 * h->d : nullptr;
    if (h->store16) {
        float* tmp = out;
        if (mem == B2IP_MEM_HOST) {
            RC_TRY(ensure(h, h->stage, static_cast<size_t>(n) * h->d * sizeof(float)));
            tmp = static_cast<float*>(h->stage.p);
        }
        widen_16bit_rows_kernel<<<h->sm_count * 8, 256, 0, h->stream>>>(h->x16, row0, n, h->d, h->d_pad, tmp, h->sh);
        if (mem == B2IP_MEM_DEVICE) { CU_TRY(h, cudaStreamSynchronize(h->stream)); return B2IP_OK; }
        src = tmp;
    }
    if (mem == B2IP_MEM_HOST) return device_to_host(h, out, src, static_cast<size_t>(n) * h->d * sizeof(float));
    CU_TRY(h, cudaMemcpyAsync(out, src, static_cast<size_t>(n) * h->d * sizeof(float),
                              cudaMemcpyDeviceToDevice, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    return B2IP_OK;
}

int b2ip_copy_to_device(b2ip_handle h, void* dst_device, const void* src_host, int64_t bytes) {
    if (!h) return B2IP_ERR_INVALID;
    if (bytes < 0 || (bytes > 0 && (!dst_device || !src_host))) return fail(h, B2IP_ERR_INVALID, "b2ip_copy_to_device: bad arguments");
    if (bytes == 0) return B2IP_OK;
    Guard g(h->device);
    RC_TRY(host_to_device(h, dst_device, src_host, static_cast<size_t>(bytes)));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    return B2IP_OK;
}

int b2ip_copy_to_host(b2ip_handle h, void* dst_host, const void* src_device, int64_t bytes) {
    if (!h) return B2IP_ERR_INVALID;
    if (bytes < 0 || (bytes > 0 && (!dst_host || !src_device))) return fail(h, B2IP_ERR_INVALID, "b2ip_copy_to_host: bad arguments");
    if (bytes == 0) return B2IP_OK;
    Guard g(h->device);
    return device_to_host(h, dst_host, src_device, static_cast<size_t>(bytes));
}

int b2ip_stats(b2ip_handle h, b2ip_stats_t* out) {
    if (!h || !out) return B2IP_ERR_INVALID;
    if (h->timing_pending) {
        Guard g(h->device);
        float ms_sum = 0.f, ref_sum = 0.f, fin_sum = 0.f, ms = 0.f;
        for (size_t i = 0; i + 3 <= h->timing_events; i += 3) {
            if (cudaEventElapsedTime(&ms, h->ev_pool[i], h->ev_pool[i + 1]) == cudaSuccess) ms_sum += ms;
            if (cudaEventElapsedTime(&ms, h->ev_pool[i + 1], h->ev_pool[i + 2]) == cudaSuccess) ref_sum += ms;
        }
        for (int b = 0; b < h->stats.query_batches; b++)
            if (cudaEventElapsedTime(&ms, h->ev_fin[2 * b], h->ev_fin[2 * b + 1]) == cudaSuccess) fin_sum += ms;
        if (cudaEventElapsedTime(&ms, h->ev_t0, h->ev_t1) == cudaSuccess) h->stats.total_ms = ms;
        cudaGetLastError();
        h->stats.coarse_ms = ms_sum;
        h->stats.refresh_ms = ref_sum;
        h->stats.finalize_ms = fin_sum;
        h->timing_pending = false;
    }
    *out = h->stats;
    return B2IP_OK;
}

const char* b2ip_last_error(b2ip_handle h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int b2ip_debug_plan_bootstrap(int64_t n_rows, int k, int cap, int sm_count, int d_pad, int max_mb,
                              int* grid, int64_t* tiles) {
    if (!grid || !tiles) return B2IP_ERR_INVALID;
    plan_bootstrap(n_rows, k, cap, sm_count, d_pad, max_mb, grid, tiles);
    return B2IP_OK;
}

int b2ip_debug_coarse_scores(b2ip_handle h, int64_t nq, const float* queries_dev, int64_t row0,
                             int64_t n_rows, float* out_dev) {
    if (!h || nq <= 0 || !queries_dev || !out_dev || row0 < 0 || n_rows <= 0 || row0 + n_rows > h->n)
        return fail(h, B2IP_ERR_INVALID, "b2ip_debug_coarse_scores: bad arguments");
    if (row0 % TILE_X != 0) return fail(h, B2IP_ERR_INVALID, "row0 must be a multiple of %d", TILE_X);
    Guard g(h->device);
    RC_TRY(ensure(h, h->q16, static_cast<size_t>(pad_q(nq)) * h->d_pad * 2));
    RC_TRY(ensure(h, h->eps2, nq * sizeof(float)));
    RC_TRY(ensure(h, h->thr, nq * sizeof(float)));
    RC_TRY(ensure(h, h->cnt, nq * sizeof(int)));
    RC_TRY(ensure(h, h->kept, nq * sizeof(int)));
    RC_TRY(ensure(h, h->flags, nq * sizeof(int)));
    prep_queries_kernel<<<static_cast<int>((pad_q(nq) + 7) / 8), 256, 0, h->stream>>>(
        queries_dev, reinterpret_cast<__nv_bfloat16*>(h->q16.p), static_cast<int>(nq), h->d, h->d_pad,
        h->norm_stats, reinterpret_cast<float*>(h->eps2.p), reinterpret_cast<float*>(h->thr.p),
        reinterpret_cast<int*>(h->cnt.p), reinterpret_cast<int*>(h->kept.p), reinterpret_cast<int*>(h->flags.p), h->sh,
        static_cast<int>(pad_q(nq)), nullptr, 0, nullptr);
    CUtensorMap tmap_q, tmap_x;
    RC_TRY(make_tmap_bf16(h, &tmap_q, h->q16.p, pad_q(nq), h->d_pad, TILE_Q));
    RC_TRY(make_tmap_bf16(h, &tmap_x, h->x16, h->n, h->d_pad, TILE_X));
    CoarseParams cp{};
    cp.num_k_blocks = h->d_pad / KBLOCK_ELEMS;
    cp.q_tiles = static_cast<int>((nq + TILE_Q - 1) / TILE_Q);
    cp.x_tiles = static_cast<int>((n_rows + TILE_X - 1) / TILE_X);
    cp.gx = h->gx;
    cp.nq = static_cast<int>(nq);
    cp.x_row0 = row0;
    cp.x_row_end = row0 + n_rows;
    cp.thr = nullptr; cp.cand = nullptr; cp.cnt = nullptr; cp.cap = 0;
    cp.dump = out_dev;
    cp.dump_ld = n_rows;
    cp.hint_q = hint_policy(h->hint_q);
    cp.hint_x = hint_policy(h->hint_x);
    cp.idesc = IDESC_SINGLE[h->sh];
    cp.dense = 0;
    const long long tiles = static_cast<long long>(cp.q_tiles) * cp.x_tiles;
    const int grid = static_cast<int>(std::min<long long>(tiles, h->sm_count));
    coarse_filter_kernel<true><<<grid, COARSE_THREADS, COARSE_SMEM_BYTES, h->stream>>>(tmap_q, tmap_x, cp);
    CU_TRY(h, cudaGetLastError());
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    return B2IP_OK;
}

}  // extern "C"
