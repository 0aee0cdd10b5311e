/*
 * b2ip.h -- C ABI of libb2ip.so, the B200 (sm_100a) exact inner-product top-k engine.
 *
 * This is the boundary a maintainer of the reference binds instead of faiss: every entry
 * point below replaces one faiss call made by the reference's `Indexer`
 * (reference src/index.py) -- the citation on each function is the call it stands in for.
 * Plain pointers and sizes only; no torch / C++ types cross the ABI; no exceptions.
 *
 * Conventions
 *   - every function returns B2IP_OK (0) or a negative B2IP_ERR_* code; the message is
 *     available from b2ip_last_error(handle) (or b2ip_last_error(NULL) for create()).
 *   - the library owns all device memory it allocates; caller buffers are borrowed for the
 *     duration of one call and every call is synchronous on return.
 *   - `mem` says where a caller buffer lives: B2IP_MEM_HOST or B2IP_MEM_DEVICE (a pointer
 *     valid on the index's device, e.g. a torch CUDA tensor's data_ptr()).
 *   - one handle = one GPU = one row shard.  Not re-entrant per handle (the reference is
 *     single-threaded); distinct handles are independent.
 *   - there is NO CPU fallback: without a CUDA device b2ip_create() fails.
 */
#ifndef B2IP_H_
#define B2IP_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct b2ip_index_s* b2ip_handle;

enum {
    B2IP_OK = 0,
    B2IP_ERR_INVALID = -1,     /* bad argument */
    B2IP_ERR_CUDA = -2,        /* CUDA runtime / driver error */
    B2IP_ERR_OOM = -3,         /* device allocation failed */
    B2IP_ERR_UNSUPPORTED = -4, /* e.g. k above B2IP_MAX_K */
    B2IP_ERR_INTERNAL = -5
};

enum { B2IP_F32 = 0, B2IP_F16 = 1, B2IP_BF16 = 2 };   /* element type of rows handed to b2ip_add */
/* how the index keeps its rows in HBM */
enum {
    B2IP_STORE_F32 = 0,  /* fp32 master rows (+ a 16-bit shadow for the coarse pass): faiss semantics */
    B2IP_STORE_F16 = 1,  /* rows ARE fp16: LOSSLESS for the reference's default pipeline, whose
                            embedding shards are float16 (generate_passage_embeddings.py:75-76)
                            and only widened by astype('float32') (src/index.py:27); fp32 rows
                            are rounded to nearest (saturating) at ingest.  A third of the
                            memory of B2IP_STORE_F32, same results on fp16-valued rows.        */
    B2IP_STORE_BF16 = 2  /* rows ARE bf16 (rounded to nearest at ingest unless given as bf16); the
                            search is exact w.r.t. those stored values, rescored in fp32 (BASELINE
                            config 4).  Half the memory, no shadow copy.                        */
};
enum { B2IP_MEM_HOST = 0, B2IP_MEM_DEVICE = 1 };

/* search strategy */
enum {
    B2IP_MODE_AUTO = 0,   /* = B2IP_MODE_TENSOR (queries whose candidate list overflows are re-run exactly) */
    B2IP_MODE_TENSOR = 1, /* tcgen05 bf16 coarse GEMM + fused threshold filter, fp32 rescore */
    B2IP_MODE_EXACT = 2   /* fp32 FMA scores + radix select (also the overflow fallback) */
};

#define B2IP_MAX_K 2048
#define B2IP_MAX_D 4096

/* Counters of the most recent b2ip_search on a handle (timings from CUDA events on the
 * handle's stream). */
typedef struct b2ip_stats_s {
    int64_t nq, ntotal;
    int32_t k, mode_used;
    int32_t coarse_launches;     /* launches of the tcgen05 scoring kernel                */
    int32_t total_launches;      /* all kernels launched by the search                    */
    float coarse_ms;             /* sum of the scoring-kernel durations                   */
    float total_ms;              /* whole device-side search                              */
    double coarse_flops;         /* 2*nq*rows*d summed over scoring launches (algorithmic) */
    int64_t candidates;          /* (query,row) pairs that passed the fused filter        */
    int64_t rescored;            /* pairs rescored in fp32                                */
    int64_t fallback_queries;    /* queries re-run on the exact path (buffer overflow)    */
    int32_t slabs;               /* corpus slabs (threshold refresh points)               */
    int32_t query_batches;
    float refresh_ms;            /* sum of the threshold-refresh kernel durations          */
    float finalize_ms;           /* rescore + final select/sort kernel durations           */
    /* run-time certificate of the coarse pass's a-priori error bound eps_q: over every row the
     * search rescored, max |coarse - exact| / eps_q (must stay < 1) and the number of rows above 1 */
    double max_err_over_eps;
    int64_t bound_violations;
    /* small batches replay their fixed launch sequence from a CUDA graph: 0 = plain launches,
     * 1 = captured by this call, 2 = replayed */
    int32_t graph_mode;
    /* batches of <= 64 queries: rows of the corpus sample whose group maxima gave the first threshold
     * (one group-max launch + one filtered slab over all rows); 0 = geometric slab schedule */
    int32_t sample_rows;
} b2ip_stats_t;

/* replaces faiss.IndexFlatIP(vector_sz)                       -- src/index.py:21
 * d: vector dimension (multiple of 4, <= 4096); device: CUDA ordinal. */
int b2ip_create(int d, int device, b2ip_handle* out);

/* Same with an explicit storage type (B2IP_STORE_*); b2ip_create == B2IP_STORE_F32. */
int b2ip_create_ex(int d, int device, int store_dtype, b2ip_handle* out);

/* drops the index and all device memory (the reference relies on GC). */
void b2ip_destroy(b2ip_handle h);

/* Run all device work of this handle on the given cudaStream_t (NULL = the handle's own
 * stream).  Lets a torch caller keep its current stream ordering. */
int b2ip_set_stream(b2ip_handle h, void* cuda_stream);

/* Tuning knobs (all have working defaults): "gx" x-tiles per raster group, "hint_q"/"hint_x"
 * L2 eviction priority of the query / corpus TMA streams (0 normal, 1 first, 2 last),
 * "cand_budget_mb" device memory allowed for candidate lists (sets the query batch),
 * "shadow_f16" (B2IP_STORE_F32 only, before the first add): 1 = fp16 operands for the coarse
 * pass instead of bf16 (tighter error bound, saturating at +-65504), "pair" 0/1 CTA-pair kernel,
 * "graph" 0/1 CUDA-graph replay of small-batch searches (env B2IP_GRAPH), "graph_timing" 0/1 keep
 * the per-kernel event records inside the graph (b2ip_stats' coarse_ms etc.), "stream_kernel" 0/1
 * streaming kernel for batches <= 64, "bootstrap" 0/1 (env B2IP_BOOTSTRAP, default 1) first
 * threshold of a batch <= 64 from the group maxima of a corpus sample + ONE filtered slab over all
 * rows instead of the geometric slab schedule, taken while the sample is at most
 * "bootstrap_max_mb" (env B2IP_BOOTSTRAP_MAX_MB, default 64) MiB of 16-bit rows (same results;
 * DESIGN.md 4.1e; b2ip_stats_t.sample_rows tells which schedule ran). */
int b2ip_set_option(b2ip_handle h, const char* name, int64_t value);

/* Optional capacity hint before a series of b2ip_add calls (avoids regrowth copies). */
int b2ip_reserve(b2ip_handle h, int64_t n_rows);

/* replaces index.add(embeddings) after embeddings.astype('float32') -- src/index.py:27,30
 * Appends n rows ([n,d] row-major, C-contiguous) of type src_dtype; rows get consecutive
 * local ids ntotal .. ntotal+n-1.  fp16 input is widened exactly, as astype does. */
int b2ip_add(b2ip_handle h, int64_t n, const void* rows, int src_dtype, int mem);

/* replaces index.ntotal                                        -- src/index.py:67-68 */
int64_t b2ip_ntotal(b2ip_handle h);
int b2ip_dim(b2ip_handle h);

/* Ids reported by b2ip_search are local row + offset (row-sharded multi-GPU: shard g
 * passes the number of rows held by shards 0..g-1). Default 0. */
int b2ip_set_row_offset(b2ip_handle h, int64_t offset);

/* A shard made of several global row ranges (e.g. every G-th ingest chunk): segment i holds
 * local rows [local_start[i], local_start[i+1]) = global rows global_start[i] + ...; both
 * arrays strictly increasing, local_start[0] = 0.  Reported ids are then global without any
 * post-processing; n_segments = 0 returns to b2ip_set_row_offset's single offset. */
int b2ip_set_row_segments(b2ip_handle h, int n_segments, const int64_t* local_start,
                          const int64_t* global_start);

/* replaces scores, indexes = index.search(q, top_docs)         -- src/index.py:42
 * queries [nq,d] fp32; out_scores [nq,k] fp32, per row descending; out_rows [nq,k] int64
 * 0-based insertion-order ids (+ row offset).  Exact ties keep the lower row.  When fewer
 * than k rows exist the tail is (-FLT_MAX, -1) as faiss pads.  NaN scores are never
 * returned.  1 <= k <= B2IP_MAX_K. */
int b2ip_search(b2ip_handle h, int64_t nq, const float* queries, int k, float* out_scores,
                int64_t* out_rows, int mode, int mem);

/* Same with the queries' element type stated: B2IP_F32 or B2IP_F16.  The reference's default
 * pipeline hands float16 query embeddings (passage_retrieval.py:154-155) to
 * `query_vectors.astype('float32')` (src/index.py:35); float16 queries are widened on the GPU
 * instead (exact, so results are identical) -- no host pass, half the host->device bytes. */
int b2ip_search_ex(b2ip_handle h, int64_t nq, const void* queries, int q_dtype, int k,
                   float* out_scores, int64_t* out_rows, int mode, int mem);

/* The one exchange step of the row-sharded search: merges n_lists per-shard results
 * (scores [n_lists,nq,k] descending per list, rows [n_lists,nq,k] global ids, -1 padded)
 * into the global top-k (score desc, ties -> lower row).  All pointers are DEVICE
 * pointers on `device`; runs on `cuda_stream` and synchronises it before returning. */
int b2ip_merge_topk(int device, void* cuda_stream, int64_t nq, int k, int n_lists,
                    const float* scores, const int64_t* rows, float* out_scores,
                    int64_t* out_rows);

/* Same, for lists that are not back to back: list l's scores start at scores +
 * l*scores_list_stride (floats), its rows at rows + l*rows_list_stride (int64s).  Lets every
 * rank all-gather ONE packed buffer per search ([rows | scores] per rank) and merge in place. */
int b2ip_merge_topk_strided(int device, void* cuda_stream, int64_t nq, int k, int n_lists,
                            const float* scores, const int64_t* rows, int64_t scores_list_stride,
                            int64_t rows_list_stride, float* out_scores, int64_t* out_rows);

/* The same exchange fused behind the search, over peer memory instead of a collective call.
 * Every rank owns a `gather` buffer of `world` slots ([rows int64 nq*k | scores fp32 nq*k],
 * slot_bytes apart) and a flag array uint32[4*world], both mapped into every other rank's address
 * space (CUDA IPC / torch symmetric memory, or plain peer access inside one process; NVLink
 * P2P).  b2ip_search_exchange runs the local
 * search with its finalize kernel storing this rank's [nq,k] block straight into slot `rank` of
 * EVERY rank's gather buffer, publishes flags[p][4*rank] = seq on every rank p, and merges the
 * world's blocks out of its own gather buffer as soon as all flags are in -- two launches queued
 * behind the search on the same stream, no host round trip and no separate all-gather.
 * Callers alternate between two buffer sets (seq parity): a rank can run at most one search
 * ahead of its slowest peer.  *status = total number of queries, over all ranks, whose candidate
 * lists overflowed (identical on every rank): when non-zero the merged output is not valid and
 * every rank must repeat the search through b2ip_search + all-gather + b2ip_merge_topk.
 *
 * Two refinements remove the per-rank work that would otherwise not shrink with the number of GPUs:
 *   - global threshold (gthr != NULL): after its last corpus slab every rank stores, per query, its
 *     ceil(k/world)-th largest coarse score into EVERY rank's threshold buffer gthr[p] (float
 *     [world][thr_stride], row = publishing rank) and raises a second flag; the minimum over ranks is
 *     a lower bound on the GLOBAL k-th coarse score, so each rank rescores only its candidates above
 *     that bound minus the error margin (about k/world + a few rows instead of k + a window).
 *   - B2IP_GATHER_OWNER: query q belongs to rank q / ceil(nq/world); a rank's block for q is stored
 *     only into the owner's gather buffer, the owner alone merges it, and out_scores/out_rows hold
 *     just the owned queries [q_lo, q_hi) compactly ([q_hi-q_lo, k]).  B2IP_GATHER_ALL: every rank
 *     receives and merges everything (out buffers [nq,k]).
 * flags[p] is uint32[4*world]: per publishing rank {results seq, overflow count, thresholds seq, 0}.
 * A flag that does not arrive within B2IP_EXCHANGE_TIMEOUT_S (environment, default 600 s) makes the
 * call fail with B2IP_ERR_INTERNAL: treat it like a collective timeout (the process group is dead).
 * All pointers are device pointers valid on the handle's device; queries [nq,d] fp32. */
#define B2IP_MAX_PEERS 8
enum { B2IP_GATHER_ALL = 0, B2IP_GATHER_OWNER = 1 };
typedef struct b2ip_exchange_s {
    int32_t world, rank;
    int64_t slot_bytes;
    void* gather[B2IP_MAX_PEERS];   /* gather[p]: rank p's gather buffer of this parity */
    void* flags[B2IP_MAX_PEERS];    /* flags[p]:  rank p's uint32[4*world] flag array of this parity */
    void* gthr[B2IP_MAX_PEERS];     /* gthr[p]:   rank p's float[world*thr_stride] threshold buffer, or all NULL */
    int64_t thr_stride;             /* floats per publishing rank in gthr (>= nq) */
    int32_t gather_mode;            /* B2IP_GATHER_ALL / B2IP_GATHER_OWNER */
    int32_t reserved;
} b2ip_exchange_t;
int b2ip_search_exchange(b2ip_handle h, int64_t nq, const float* queries_dev, int k,
                         const b2ip_exchange_t* ex, uint32_t seq, float* out_scores_dev,
                         int64_t* out_rows_dev, int64_t* status);

/* One process driving several GPUs (the reference driver is a single process): lets kernels of
 * this handle's device store into buffers that live on `peer_device` (cudaDeviceEnablePeerAccess),
 * so b2ip_search_exchange can be used between handles of the same process with plain device
 * pointers in b2ip_exchange_t.  Fails with B2IP_ERR_UNSUPPORTED when the devices have no P2P path. */
int b2ip_enable_peer_access(b2ip_handle h, int peer_device);

/* The row-sharded search of ONE process over several handles (one per GPU, each holding a row
 * shard whose ids are made global with b2ip_set_row_offset / b2ip_set_row_segments): what the
 * reference's single-process driver (passage_retrieval.py never starts torch.distributed) needs to
 * use a whole multi-GPU box.  b2ip_group_search takes HOST queries ([nq,d] fp32 or fp16) and fills
 * HOST results ([nq,k]); inside, one worker thread per member uploads the queries, runs
 * b2ip_search_exchange (global threshold, owner mode) against library-owned peer buffers and
 * downloads the slice of queries its GPU owns -- uploads, searches and downloads of all members
 * overlap, no Python in between.  *status != 0: a candidate list overflowed somewhere, the output
 * is not valid and the caller repeats the search member by member (b2ip_search + b2ip_merge_topk).
 * The handles must outlive the group; a group is not re-entrant. */
typedef struct b2ip_group_s* b2ip_group;
int b2ip_group_create(int n_handles, const b2ip_handle* handles, b2ip_group* out);
void b2ip_group_destroy(b2ip_group g);
int b2ip_group_search(b2ip_group g, int64_t nq, const void* queries_host, int q_dtype, int k,
                      float* out_scores_host, int64_t* out_rows_host, int64_t* status);
const char* b2ip_group_last_error(b2ip_group g);

/* replaces faiss.write_index's read of the stored vectors       -- src/index.py:53
 * Copies rows [row0, row0+n) as fp32 into out ([n,d]). */
int b2ip_export_rows(b2ip_handle h, int64_t row0, int64_t n, float* out, int mem);

/* Host <-> device copies through the handle's pinned double-buffered staging (a pool of copy
 * threads fills / drains two page-locked buffers while the copy engine moves the other one):
 * what b2ip_add / b2ip_search use for pageable host buffers, exposed for callers that keep
 * queries or results in their own device buffers (the single-process multi-GPU Indexer uploads
 * the queries once and fans them out over NVLink).  Synchronous; `*_device` pointers must be
 * valid on the handle's device. */
int b2ip_copy_to_device(b2ip_handle h, void* dst_device, const void* src_host, int64_t bytes);
int b2ip_copy_to_host(b2ip_handle h, void* dst_host, const void* src_device, int64_t bytes);

int b2ip_stats(b2ip_handle h, b2ip_stats_t* out);
const char* b2ip_last_error(b2ip_handle h);

/* Test hook: raw bf16 tensor-core scores of queries [nq,d] (device fp32) against rows
 * [row0,row0+n_rows) written to out [nq,n_rows] (device fp32) by the same tcgen05
 * mainloop the search uses (filter replaced by a store). */
int b2ip_debug_coarse_scores(b2ip_handle h, int64_t nq, const float* queries_dev, int64_t row0,
                             int64_t n_rows, float* out_dev);

/* Test hook, host arithmetic only (no CUDA call: usable without a GPU): the corpus sample a batch of
 * <= 64 queries would take its first threshold from -- *grid CTAs over *tiles tiles of 128 rows --
 * on a shard of n_rows rows for the given k, list capacity, SM count, padded dimension and
 * "bootstrap_max_mb"; *grid = 0 when the geometric slab schedule is kept (DESIGN.md 4.1e). */
int b2ip_debug_plan_bootstrap(int64_t n_rows, int k, int cap, int sm_count, int d_pad, int max_mb,
                              int* grid, int64_t* tiles);

/* Library build info: "b2ip <version> sm_100a ..." */
const char* b2ip_version(void);

#ifdef __cplusplus
}
#endif
#endif /* B2IP_H_ */
