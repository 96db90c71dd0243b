// Internal definitions shared by the engine's translation units (not part of the C ABI).
#pragma once
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>

#include <algorithm>
#include <array>
#include <cstdint>
#include <cstdio>
#include <atomic>
#include <map>
#include <memory>
#include <string>
#include <tuple>
#include <unordered_map>
#include <unordered_set>
#include <utility>
#include <vector>

#include "pemspgemm.h"

// ---------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------
enum { PEM_NSCALARS = 24, PEM_NEVENTS = 8, PEM_PLAN_MAX = 96 };

// Sizes a product read back from the device (tile products, kept pairs, C' tiles, nnz ...), in program order.
// A repeated product of the same operands replays them instead of stalling the host at every read-back: the
// kernels still compute every size on the device, the copies are only compared after the product's final sync
// (a mismatch cannot happen: a handle's pattern is immutable, only its values may be refreshed; if it does, the
// product is redone with the stalls).
struct pem_graph;
struct pem_plan {
    int64_t v[PEM_PLAN_MAX];
    int n = 0;
    bool valid = false;
    // PEM_OPT_GRAPHS: the replayed product captured as one CUDA graph over buffers the graph owns (spgemm.cu)
    std::shared_ptr<pem_graph> graph;
    bool graph_failed = false;      // the capture was tried and given up (a host stall inside, or over the memory budget)
    size_t alloc_bytes = 0;         // bytes the recording product asked the allocator for: upper bound of a graph's arena
};
// pairs per block of step 2's pair kernel; step 1 (k_ctiles) emits the first tile of every such block
constexpr int PEM_PAIR_BLOCK = 128;

// kernels timed individually (CUDA events on the context's stream) for the roofline report
enum { KT_EXPAND = 0, KT_SORT = 1, KT_PAIRS = 2, KT_NUMERIC = 3, KT_N = 4 };

struct pem_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;   // host->device copy of the values, overlapped with key generation and the sort
    cudaEvent_t ev_copy[2] = {};
    cudaMemPool_t pool = nullptr;
    std::string err;
    int64_t launches = 0;        // kernels of this library launched on the stream
    int last_step3_kernel = 0;   // step 3 of the last product: 1 = row-owner, 2 = entry-owner, 3 = tile-class, 4 = window kernel
    int last_sort_passes = -1;   // step 1 of the last product: -1 = no sort (bitmap path), 0 = block-local row sort, n = n radix passes
    int opt_keep_empty = 0;      // PEM_OPT_KEEP_EMPTY_TILES
    int opt_step1_path = 0;      // PEM_OPT_STEP1_PATH
    int opt_owner = 0;           // PEM_OPT_OWNER: 0 = automatic (window or entry-owner), 2 = entry-owner, 1 = row-owner (registers), 3 = tile-class kernel, 4 = window kernel
    int opt_trace = 0;           // PEM_OPT_TRACE: host-side timeline of step 1 on stderr
    int opt_esc_variant = 0;     // PEM_OPT_ESC_VARIANT: bit 0 = count-then-write expansion, bit 1 = no block-local row sort
    int opt_step2_kernel = 0;    // PEM_OPT_STEP2_KERNEL: 0 = lane per pair (list or row-mask form by tile density), 1 = list form, 3 = row-mask form, 2 = sixteen lanes per C' tile
    int opt_async_vals = 0;      // PEM_OPT_ASYNC_VALUES: pem_convert_coo returns while the values' upload is still in flight
    int opt_s3_small_e = 8;      // PEM_OPT_S3_SMALL_NNZ: step 3 handles a tile with at most this many nonzeros ...
    int opt_s3_small_np = 64;    // PEM_OPT_S3_SMALL_PAIRS: ... and at most this many pairs with one thread
    int opt_poison = 0;          // PEM_OPT_POISON: 0 or 0x100 | byte every allocated block is filled with (tests)
    int sm_count = 148;
    int smem_optin = 227 * 1024; // max dynamic shared memory per block
    int64_t* h_scalars = nullptr; // pinned, PEM_NSCALARS entries: size read-backs
    int64_t* h_check = nullptr;   // pinned, PEM_PLAN_MAX entries: the same read-backs of a replayed product, compared at its end
    std::map<std::vector<int64_t>, pem_plan> plans;   // key: operand ids, panel, options that change sizes
    pem_plan* plan = nullptr;     // plan of the product in flight (pem_spgemm_panel only; stage-level calls stall)
    bool plan_replay = false;
    int plan_pos = 0;
    int opt_plans = 1;            // PEM_OPT_SIZE_PLANS
    int opt_graphs = 1;           // PEM_OPT_GRAPHS: repeats of a product run as one captured CUDA graph
    pem_graph* cap = nullptr;     // graph being captured: allocations come from / go back to its arena
    size_t graph_bytes = 0, graph_limit = (size_t)8 << 30;   // bytes held by graph arenas / their budget (a quarter of the memory free at creation)
    int64_t graph_replays = 0;    // products that ran as a graph launch since creation (pem_ctx_graph_replays)
    size_t prod_alloc = 0;        // bytes requested from the allocator by the product in flight
    int64_t size_stalls = 0;      // host stalls at size read-backs since creation (pem_ctx_size_stalls)
    int64_t* d_scalars = nullptr; // device mirror the kernels reduce into
    cudaEvent_t ev[PEM_NEVENTS] = {};
    cudaEvent_t kev[2 * KT_N] = {};   // begin/end pairs of the individually timed kernels
    bool kt_seen[KT_N] = {};
    double kt_ms[KT_N] = {};          // resolved by pem_spgemm_panel after its final sync
    // caching layer over the pool: freed blocks are kept by size and handed out again in stream
    // order (all work of a context is on one stream), so a repeated SpGEMM allocates nothing
    std::multimap<size_t, void*> free_blocks;
    std::unordered_map<void*, size_t> live_blocks;
    size_t cached_bytes = 0, cache_limit = (size_t)32 << 30;
    int64_t pool_mallocs = 0;    // cudaMallocFromPoolAsync calls (cache misses) since creation
    size_t pool_taken = 0;       // bytes this context holds from its pool (live + cached)
    size_t free_at_create = 0;   // device memory free when the context was created (cudaMemGetInfo costs ~1 ms: never on the hot path)

    int fail(int code, const std::string& msg) { err = msg; return code; }
    int fail_cuda(cudaError_t e, const char* what, const char* file, int line)
    {
        char buf[512];
        snprintf(buf, sizeof buf, "CUDA error %d (%s) at %s:%d: %s", (int)e, cudaGetErrorString(e), file, line, what);
        err = buf;
        (void)cudaGetLastError();
        return PEM_ERR_CUDA;
    }
};

// NVTX range around a stage (shows up in Nsight Systems / ncu --nvtx; a no-op without a tool attached)
struct PemRange {
    explicit PemRange(const char* name) { nvtxRangePushA(name); }
    ~PemRange() { nvtxRangePop(); }
};
#define PEM_RANGE(name) PemRange pem_range__(name)

#define PEM_CK(call)                                                                     \
    do {                                                                                 \
        cudaError_t e__ = (call);                                                        \
        if (e__ != cudaSuccess) return ctx->fail_cuda(e__, #call, __FILE__, __LINE__);   \
    } while (0)

// kernel launch check + launch accounting
#define PEM_LAUNCHED()                                                                   \
    do {                                                                                 \
        ++ctx->launches;                                                                 \
        cudaError_t e__ = cudaGetLastError();                                            \
        if (e__ != cudaSuccess) return ctx->fail_cuda(e__, "kernel launch", __FILE__, __LINE__); \
    } while (0)

// timing events: inside a graph capture they become event-record nodes that record on every launch of the graph
static inline cudaError_t pem_event_record(pem_ctx* ctx, cudaEvent_t ev)
{
    return cudaEventRecordWithFlags(ev, ctx->stream, ctx->cap ? cudaEventRecordExternal : cudaEventRecordDefault);
}
#define KT_BEGIN(id) do { pem_event_record(ctx, ctx->kev[2 * (id)]); } while (0)
#define KT_END(id) do { pem_event_record(ctx, ctx->kev[2 * (id) + 1]); ctx->kt_seen[id] = true; } while (0)

#define PEM_TRY(expr)                    \
    do {                                 \
        int rc__ = (expr);               \
        if (rc__ != PEM_OK) return rc__; \
    } while (0)

// stream-ordered allocation from the context's pool through the caching layer
// (never returns a null pointer for n == 0)
int pem_alloc_bytes(pem_ctx* ctx, void** p, size_t bytes);
void pem_free_bytes(pem_ctx* ctx, void* p);
void pem_cache_release(pem_ctx* ctx);
template <class T>
static inline int pem_alloc(pem_ctx* ctx, T** p, size_t n)
{
    return pem_alloc_bytes(ctx, (void**)p, (n ? n : 1) * sizeof(T));
}
template <class T>
static inline void pem_free(pem_ctx* ctx, T*& p)
{
    if (p) pem_free_bytes(ctx, (void*)p);
    p = nullptr;
}

// local temporaries that go back to the cache on EVERY return path (the PEM_TRY / PEM_CK early returns included):
// `pem_guard g(ctx, keys, pos, tmp);`.  Whatever is still held at a return is freed there, in the order listed; a
// block the code is done with earlier keeps its explicit pem_free, which nulls the pointer, so nothing is freed twice
template <class... T>
struct pem_guard {
    pem_ctx* ctx;
    std::tuple<T*&...> p;
    explicit pem_guard(pem_ctx* c, T*&... q) : ctx(c), p(q...) {}
    ~pem_guard() { std::apply([this](auto&... q) { (pem_free(ctx, q), ...); }, p); }
    pem_guard(const pem_guard&) = delete;
    pem_guard& operator=(const pem_guard&) = delete;
};

static inline uint64_t pem_next_uid()
{
    static std::atomic<uint64_t> next{1};
    return next.fetch_add(1);
}

static inline int pem_div_up(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

// ---------------------------------------------------------------------------------------
// tiled matrix (SURVEY.md 2.2; arrays named after the reference's)
// ---------------------------------------------------------------------------------------
// value type of a tiled matrix / result: the reference is fp64 only (spgemm.cu:728, `ValueType`, a template
// parameter there); fp32 is the second instantiation SURVEY.md section 8f rank 4 asks for.  The `vals`
// pointers below are typed double* and reinterpreted as float* when dtype == PEM_F32.
enum { PEM_F64 = 0, PEM_F32 = 1 };
static inline size_t pem_vsize(int dtype) { return dtype == PEM_F32 ? 4 : 8; }

// A launch written once for both value types: launch(float{}) or launch(double{}) by dtype, the lambda taking the type
// as `using VT = decltype(v)`; pem_vals<VT> views a value array (double* in the handles, void* at the ABI) as VT.
template <class F>
static inline void pem_by_dtype(int dtype, F&& launch)
{
    if (dtype == PEM_F32) launch(float{});
    else launch(double{});
}
template <class V> static inline V* pem_vals(void* p) { return static_cast<V*>(p); }
template <class V> static inline const V* pem_vals(const void* p) { return static_cast<const V*>(p); }

// What built a tiled matrix: the entry points that rewrite its values from the same sources accept those only
enum { PEM_BUILT_INPUT = 0, PEM_BUILT_RESULT = 1, PEM_BUILT_SUM = 2 };
struct pem_origin {
    int kind = PEM_BUILT_INPUT;       // conversion or transpose: new values come through pem_tiled_set_values
    uint64_t a_uid = 0, b_uid = 0;    // result: the operands of its product; sum: A and B, in that order
    int32_t rb = 0, re = 0;           // result: its panel
};

struct pem_tiled {
    uint64_t uid = 0;                 // unique per conversion (the pattern is immutable, the values may be refreshed): key of the size plans
    int dtype = PEM_F64;
    int32_t rows = 0, cols = 0;
    int64_t nnz = 0;
    int32_t tile_rows = 0, tile_cols = 0, tiles = 0;
    double* vals = nullptr;           // [nnz] tile-major, row-major inside a tile
    uint32_t* tile_nnz_ptr = nullptr; // [tiles+1]
    uint16_t* masks = nullptr;        // [tiles*16] row masks
    uint16_t* masks_t = nullptr;      // [tiles*16] column masks
    uint8_t* row_ptr = nullptr;       // [tiles*16]
    int32_t* tile_row_ptr = nullptr;  // [tile_rows+1]
    int32_t* tile_col_idx = nullptr;  // [tiles]
    int32_t* tile_row_idx = nullptr;  // [tiles]
    uint16_t* col_occ = nullptr;      // [tiles]
    uint16_t* row_occ = nullptr;      // [tiles]
    uint8_t* rc_idx = nullptr;        // [nnz] (r<<4)|c of every value, tile-major (the reference's *tiles_rowColIdx)
    uint32_t* val_pos = nullptr;      // [nnz] index of every value slot in the input the handle was built from (pem_tiled_set_values)
    // conversion from host memory: the values' upload and their gather into tile order run on the context's
    // copy stream, BEHIND the call that returns this handle, so the symbolic steps of a product (which read
    // masks only) overlap them; whoever reads `vals` first makes the engine's stream wait (pem_tiled_wait_vals)
    cudaEvent_t ev_vals = nullptr;    // recorded on the copy stream after the gather
    bool vals_pending = false;
    void* pend_buf = nullptr;         // staging buffer the gather still reads (uploaded values)
    std::vector<int32_t> h_tile_row_ptr;  // host copy of tile_row_ptr: panel calls find their tile range without a device read
    // row slices, built on first use as a B operand of step 1 (pem_tiled_build_srow): for every
    // matrix row s the ids of the tiles that hold a nonzero of row s (in no particular order)
    int64_t* srow_ptr = nullptr;      // [rows16+1], rows16 = 16*tile_rows
    int32_t* srow_tile = nullptr;     // [srow_ptr[rows16]]
    int64_t srow_total = 0;
    // step-3 views, built on first use (pem_tiled_build_views): one 32-bit record per tile row /
    // tile column = mask | first-value offset << 16, and the values in column-major order inside a tile
    uint32_t* row_rec = nullptr;      // [tiles*16]  masks[i]   | row_ptr[i] << 16          (operand A)
    uint32_t* col_rec = nullptr;      // [tiles*16]  masks_t[i] | first value of column << 24 (operand B)
    double* vals_t = nullptr;         // [nnz] tile-major, column-major inside a tile        (operand B)
    // pem_tiled_refresh_from_result accepts results of the product (and panel) a result handle came from, whose structure
    // it holds; pem_tiled_add_values the operands of a sum.  A transpose records nothing.
    pem_origin origin;
    int2* add_src = nullptr;          // [tiles] sum S = alpha*A + beta*B: per tile of S the tile of A and of B it holds (-1: none)
    // every device array above, in the order pem_tiled_free releases them: the twelve of the structure
    // (pem_tiled_alloc_values / _tiles), the caches built on first use and a sum's source tiles
    std::array<void**, 18> buffers()
    {
        return {(void**)&vals, (void**)&tile_nnz_ptr, (void**)&masks, (void**)&masks_t, (void**)&row_ptr,
                (void**)&tile_row_ptr, (void**)&tile_col_idx, (void**)&tile_row_idx, (void**)&col_occ,
                (void**)&row_occ, (void**)&rc_idx, (void**)&val_pos, (void**)&srow_ptr, (void**)&srow_tile,
                (void**)&row_rec, (void**)&col_rec, (void**)&vals_t, (void**)&add_src};
    }
};

// A handle under construction: freed with everything it holds unless the builder releases it into *out
struct pem_tiled_deleter {
    pem_ctx* ctx;
    void operator()(pem_tiled* t) const { pem_tiled_free(ctx, t); }
};
using pem_tiled_ptr = std::unique_ptr<pem_tiled, pem_tiled_deleter>;

// A new rows x cols handle of nnz values: its own uid (the key of the size plans), its tile counts from the shape
static inline pem_tiled_ptr pem_tiled_new(pem_ctx* ctx, int dtype, int32_t rows, int32_t cols, int64_t nnz)
{
    pem_tiled_ptr T(new pem_tiled(), pem_tiled_deleter{ctx});
    T->uid = pem_next_uid();
    T->dtype = dtype;
    T->rows = rows; T->cols = cols; T->nnz = nnz;
    T->tile_rows = pem_div_up(rows, PEM_TILE);
    T->tile_cols = pem_div_up(cols, PEM_TILE);
    return T;
}
// The structure arrays of a handle: the per-value ones (vals, rc_idx, val_pos) for T->nnz values, the per-tile ones
// (tile_row_ptr included) for T->tiles tiles and T->tile_rows tile rows.  Nothing is written.
static inline int pem_tiled_alloc_values(pem_ctx* ctx, pem_tiled* T)
{
    PEM_TRY(pem_alloc_bytes(ctx, (void**)&T->vals, std::max<size_t>(1, (size_t)T->nnz * pem_vsize(T->dtype))));
    PEM_TRY(pem_alloc(ctx, &T->rc_idx, (size_t)T->nnz));
    return pem_alloc(ctx, &T->val_pos, (size_t)T->nnz);
}
static inline int pem_tiled_alloc_tiles(pem_ctx* ctx, pem_tiled* T)
{
    const size_t n = (size_t)T->tiles;
    PEM_TRY(pem_alloc(ctx, &T->tile_row_ptr, (size_t)T->tile_rows + 1)); PEM_TRY(pem_alloc(ctx, &T->tile_nnz_ptr, n + 1));
    PEM_TRY(pem_alloc(ctx, &T->masks, n * 16)); PEM_TRY(pem_alloc(ctx, &T->masks_t, n * 16));
    PEM_TRY(pem_alloc(ctx, &T->row_ptr, n * 16)); PEM_TRY(pem_alloc(ctx, &T->tile_col_idx, n));
    PEM_TRY(pem_alloc(ctx, &T->tile_row_idx, n)); PEM_TRY(pem_alloc(ctx, &T->col_occ, n));
    return pem_alloc(ctx, &T->row_occ, n);
}
static inline int pem_tiled_alloc(pem_ctx* ctx, pem_tiled* T)
{
    PEM_TRY(pem_tiled_alloc_values(ctx, T));
    return pem_tiled_alloc_tiles(ctx, T);
}
// Every builder's last step before it releases T into *out: mirror tile_row_ptr into h_tile_row_ptr (panel calls find
// their tile range there without a device read) and wait for the stream.  Read-backs the builder enqueued before are
// then on the host, for its last checks.
static inline int pem_tiled_publish(pem_ctx* ctx, pem_tiled* T)
{
    T->h_tile_row_ptr.resize((size_t)T->tile_rows + 1);
    PEM_CK(cudaMemcpyAsync(T->h_tile_row_ptr.data(), T->tile_row_ptr, ((size_t)T->tile_rows + 1) * 4,
                           cudaMemcpyDeviceToHost, ctx->stream));
    PEM_CK(cudaStreamSynchronize(ctx->stream));
    return PEM_OK;
}

// ---- value slots of a tiled matrix: k_refresh_vals, k_refresh_slots, k_col_views (convert.cu), k_add_vals (sum.cu) ----
// Slot in vals_t (column-major inside a tile) of the value in row r of a column whose record (col_rec) is cr, in the
// tile whose values start at ts: the column's first value (top byte of the record) plus the column's rows above r.
__device__ __forceinline__ uint32_t pem_col_slot(uint32_t ts, uint32_t cr, unsigned r)
{
    return ts + (cr >> 24) + __popc(cr & ((1u << r) - 1u));
}

// Writes value(x, t) into every value slot x of tile t of a tiled matrix: into vals and, when the column-major view
// exists, into vals_t.  A warp takes 32 consecutive tiles and walks their slots, which are contiguous, one per lane, so
// the (r, c) bytes and the value arrays move in whole sectors; a lane finds its tile among the warp's 32 in five
// shuffles over the tiles' first offsets, which the lanes hold in registers.  The caller passes the thread indices, read
// in the kernel, where its launch bounds limit them.
template <class T, class F>
__device__ __forceinline__ void
pem_write_slots(int64_t gid, unsigned tid, int cnt, const uint32_t* __restrict__ tile_nnz_ptr,
                const uint8_t* __restrict__ rc_idx, const uint32_t* __restrict__ col_rec, T* __restrict__ vals,
                T* __restrict__ vals_t, F value)
{
    const int64_t t0 = (gid >> 5) * 32;
    if (t0 >= cnt) return;                          // whole warps leave together
    const int lane = tid & 31;
    const int nt = (int)(cnt - t0 < 32 ? cnt - t0 : 32);
    const uint32_t first = tile_nnz_ptr[t0 + min(lane, nt)];   // lanes >= nt hold the end: above every x
    const uint32_t s = __shfl_sync(0xffffffffu, first, 0), e = tile_nnz_ptr[t0 + nt];
    for (uint32_t b = s; b < e; b += 32) {
        const uint32_t x = b + lane;
        int j = 0;                                  // last tile of the warp whose first offset is <= x
        uint32_t ts = s;
#pragma unroll
        for (int step = 16; step > 0; step >>= 1) {
            const uint32_t f = __shfl_sync(0xffffffffu, first, j + step);
            if (f <= x) { j += step; ts = f; }
        }
        if (x < e) {
            const T v = value(x, t0 + j);
            vals[x] = v;
            if (vals_t) {
                const unsigned rc = rc_idx[x];
                const unsigned r = rc >> 4, c = rc & 15u;
                const uint32_t cr = col_rec[(size_t)(t0 + j) * 16 + c];
                vals_t[pem_col_slot(ts, cr, r)] = v;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------
// result: C or a tile-row panel of C
// ---------------------------------------------------------------------------------------
struct pem_result {
    int dtype = PEM_F64;
    int32_t rb = 0, re = 0;           // panel of A' tile rows
    int32_t rows = 0, cols = 0;       // shape of the full C
    int32_t tile_cols = 0;
    int64_t tiles = 0, pairs = 0, nnz = 0, tile_products = 0;
    int stage = 0;                    // 1, 2, 3 = last completed step
    bool s3_entries = false;          // step 3 runs the entry-owner kernel (PEM_OPT_OWNER = 2)
    bool s2_pairs = false;            // step 2 ran the pair kernel (pair_hit may still be null: dense-tile mode, see pem_step2_symbolic)
    int s3_kernel = 0;                // numeric kernel step 3 ran (pem_ctx_last_step3_kernel's numbering); pem_spgemm_numeric reruns it
    uint64_t a_uid = 0, b_uid = 0;    // operands of step 1: pem_spgemm_numeric accepts these handles only
    bool keep_empty = false;          // step 1 ran under PEM_OPT_KEEP_EMPTY_TILES: C' may hold tiles with no nonzero
    int64_t* row_ptr = nullptr;       // [re-rb+1]
    int32_t* tile_row = nullptr;      // [tiles]
    int32_t* tile_col = nullptr;      // [tiles]
    int64_t* pair_ptr = nullptr;      // [tiles+1]
    int2* pair_list = nullptr;        // [pairs] (A tile id, B tile id), ascending A tile id inside a C' tile
    uint16_t* masks = nullptr;        // [tiles*16]
    int64_t* tile_nnz_ptr = nullptr;  // [tiles+1]
    uint8_t* row_col_idx = nullptr;   // [nnz], produced on demand (pem_result_make_rowcolidx)
    uint32_t* pair_hit = nullptr;     // [pairs] entry-owner variant: (C rows hit << 16) | C columns hit by the pair
    int32_t* blk_tile = nullptr;      // entry-owner variant: first tile of each 128-entry step-3 block
    int32_t* pair_blk = nullptr;      // first tile of each 256-pair step-2 block (optional by-product of step 1)
    double* vals = nullptr;           // [nnz]
    std::shared_ptr<pem_graph> graph; // set when the buffers above belong to a product graph's arena (pem_result_free hands them back to it)
    // every device buffer above, in the order pem_result_free releases them
    std::array<void**, 12> buffers()
    {
        return {(void**)&row_ptr, (void**)&tile_row, (void**)&tile_col, (void**)&pair_ptr, (void**)&pair_list,
                (void**)&pair_hit, (void**)&blk_tile, (void**)&pair_blk, (void**)&masks, (void**)&tile_nnz_ptr,
                (void**)&row_col_idx, (void**)&vals};
    }
};

// A repeated product captured as ONE CUDA graph (PEM_OPT_GRAPHS; pem_spgemm_panel).  The graph bakes device
// pointers in, so it owns every block its product touches (the arena: result buffers and temporaries): a result
// handed out from it borrows the result buffers, and the graph can run again once that result has been freed.
struct pem_graph {
    pem_ctx* ctx = nullptr;
    cudaGraphExec_t exec = nullptr;
    std::vector<std::pair<void*, size_t>> arena;   // every block taken during the capture
    std::unordered_set<void*> owned;               // the same pointers, for pem_result_free
    std::multimap<size_t, void*> idle;             // arena blocks free at the current point of the capture
    size_t bytes = 0;
    bool busy = false;                // a result borrowed from this graph is alive
    bool side_allocs = false;         // blocks came from the pool on the copy stream during the capture
    pem_result tmpl;                  // the product's result as the captured run left it
    int64_t launches = 0;             // kernels per launch of the graph
    int last_step3_kernel = 0, last_sort_passes = -1;
    bool kt_seen[KT_N] = {};
    int opts[5] = {};                 // options the kernel choice depends on (owner, step-2 kernel, small-tile limits, trace)
    ~pem_graph();
};
void pem_graph_opts(const pem_ctx* ctx, int* o);

// scalars slots in ctx->d_scalars / h_scalars
enum {
    SC_ERR = 0,       // error flags from kernels
    SC_COUNT = 1,     // generic count (tiles found by the census)
    SC_MAXWIN = 2,    // step 1: max window words over the panel's rows
    SC_MAXP = 3,      // step 1: max tile products of a row
    SC_MAXD = 4,      // step 1: max C' tiles of a row
    SC_SUMP = 5,      // step 1: total tile products
    SC_T0 = 6, SC_T1 = 7, SC_T2 = 8,
    SC_NSMALL1 = 9, SC_NLARGE1 = 10,  // step 1: rows per kernel-2 list
    SC_NSMALL2 = 11, SC_NLARGE2 = 12, // step 1: rows per kernel-3 list
    SC_WORK0 = 16                     // step 1: four work-queue cursors (count large/small, fill large/small)
};

// One host read-back of device-side sizes: add() enqueues copies, get() returns the values: after a stream
// synchronisation, or, when the product in flight replays a plan, immediately from the plan.
struct pem_size_read {
    pem_ctx* ctx;
    int n = 0;
    explicit pem_size_read(pem_ctx* c) : ctx(c) {}
    bool replay() const { return ctx->plan && ctx->plan_replay; }
    int add(const int64_t* d_src, int cnt)
    {
        if (n + cnt > PEM_NSCALARS || (ctx->plan && ctx->plan_pos + n + cnt > PEM_PLAN_MAX))
            return ctx->fail(PEM_ERR_LIMIT, "size read-back overflow");
        int64_t* dst = replay() ? ctx->h_check + ctx->plan_pos + n : ctx->h_scalars + n;
        PEM_CK(cudaMemcpyAsync(dst, d_src, (size_t)cnt * 8, cudaMemcpyDeviceToHost, ctx->stream));
        n += cnt;
        return PEM_OK;
    }
    int get(int64_t* out)
    {
        if (replay()) {
            if (ctx->plan_pos + n > ctx->plan->n) return ctx->fail(PEM_ERR_ARG, "size plan out of step");
            for (int i = 0; i < n; ++i) out[i] = ctx->plan->v[ctx->plan_pos + i];
        } else {
            PEM_CK(cudaStreamSynchronize(ctx->stream));
            ++ctx->size_stalls;
            for (int i = 0; i < n; ++i) out[i] = ctx->h_scalars[i];
            if (ctx->plan)
                for (int i = 0; i < n; ++i) ctx->plan->v[ctx->plan_pos + i] = out[i];
        }
        if (ctx->plan) ctx->plan_pos += n;
        n = 0;
        return PEM_OK;
    }
};

// step entry points implemented in spgemm.cu / convert.cu / export.cu
int pem_scan_exclusive_i64(pem_ctx* ctx, int64_t* d_inout, int64_t n);  // in place, n elements
extern "C" int pem_result_make_rowcolidx(pem_ctx* ctx, pem_result* C);
int pem_step1_esc(pem_ctx* ctx, const pem_tiled* A, const pem_tiled* B, pem_result* C);  // step1_esc.cu
int pem_tiled_build_srow(pem_ctx* ctx, const pem_tiled* B);                              // convert.cu
int pem_tiled_wait_vals(pem_ctx* ctx, const pem_tiled* T);                               // convert.cu
int pem_tiled_build_views(pem_ctx* ctx, const pem_tiled* T, bool as_a, bool as_b);       // convert.cu
int pem_tiled_write_slots(pem_ctx* ctx, pem_tiled* T, const void* dV);                   // convert.cu: V in T's slot order
int pem_operand_structure(pem_ctx* ctx, const pem_result* C, const int32_t* keep, pem_tiled* T);  // operand.cu
int pem_step3_launch(pem_ctx* ctx, const pem_tiled* A, const pem_tiled* B, pem_result* C);  // step3.cu: C->s3_kernel on C's buffers
