// Context, options, handle accessors and small shared device helpers of the C ABI.
// Replaces the ad-hoc stream / RMM pool setup of the reference (spgemm.cu:757-758,808-817) with
// one stream + one stream-ordered cudaMemPool_t whose release threshold is "never", so that
// per-iteration cudaMallocAsync/cudaFreeAsync of the C-side buffers (spgemm.cu:1138-1295,
// 1118-1131) are pool hits and leave the critical path.
#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <cstring>
#include <new>

#include "engine.cuh"

// ---- caching allocator -----------------------------------------------------------------------
// Replaces the reference's per-iteration cudaMallocAsync + 11 blocking cudaFree (spgemm.cu:1118-1131,
// 1138-1295; its malloc_time).  Blocks come from the context's cudaMemPool_t once and are then
// recycled by size: a block serves a request of up to its own size and no less than three quarters of it
// (sequential tile-row panels of one product ask for similar, not equal, sizes).  Cached blocks are
// only handed back to the driver when an allocation fails, when the cache outgrows its limit (80 % of the
// memory that was free when the context was created; PEM_OPT_CACHE_LIMIT_MB) or on pem_ctx_trim:
// unmapping and re-mapping tens of GB costs seconds, far more than any kernel here.
//
// While a product is being captured into a CUDA graph (ctx->cap, pem_spgemm_panel) every block it takes joins
// the graph's arena and stays there: freed blocks go to the arena's own idle list (later allocations of the same
// capture reuse them: the graph is one chain, so stream order holds), never back to the shared cache, because
// the graph bakes their addresses in.  A miss goes to the pool on the COPY stream (the engine's stream is
// capturing); pem_spgemm_panel drains that stream before the first launch of the graph.
//
// PEM_OPT_POISON fills every block handed out with one byte pattern, in stream order on the engine's stream, before
// the caller sees it: all of it, also the part of a cached block beyond the request.  Every user of a block runs on
// that stream or waits on an event recorded there after the allocation (the copy stream's value upload and gather
// in convert.cu), so the fill lands before the block's first use.  Inside a capture the fill is a memset node of the
// graph, so every launch of the graph poisons its arena again.
static int poison(pem_ctx* ctx, void* p, size_t bytes)
{
    if (!ctx->opt_poison || !bytes) return PEM_OK;
    PEM_CK(cudaMemsetAsync(p, ctx->opt_poison & 0xFF, bytes, ctx->stream));
    return PEM_OK;
}

static int graph_alloc_bytes(pem_ctx* ctx, void** p, size_t bytes)
{
    pem_graph& g = *ctx->cap;
    auto own = [&](void* q, size_t sz) {
        g.arena.emplace_back(q, sz);
        g.owned.insert(q);
        g.bytes += sz;
    };
    auto it = g.idle.lower_bound(bytes);
    if (it != g.idle.end() && it->first - bytes <= it->first / 4) {
        *p = it->second;
        size_t sz = it->first;
        g.idle.erase(it);
        return poison(ctx, *p, sz);
    }
    it = ctx->free_blocks.lower_bound(bytes);
    if (it != ctx->free_blocks.end() && it->first - bytes <= it->first / 4) {
        *p = it->second;
        size_t sz = it->first;
        ctx->live_blocks[*p] = sz;
        ctx->cached_bytes -= sz;
        own(*p, sz);
        ctx->free_blocks.erase(it);
        return poison(ctx, *p, sz);
    }
    cudaError_t e = cudaMallocFromPoolAsync(p, bytes, ctx->pool, ctx->copy_stream);
    if (e != cudaSuccess) return ctx->fail_cuda(e, "cudaMallocFromPoolAsync (graph arena)", __FILE__, __LINE__);
    g.side_allocs = true;
    ctx->live_blocks[*p] = bytes;
    ctx->pool_taken += bytes;
    ++ctx->pool_mallocs;
    own(*p, bytes);
    return poison(ctx, *p, bytes);
}

int pem_alloc_bytes(pem_ctx* ctx, void** p, size_t bytes)
{
    bytes = (bytes + 511) & ~(size_t)511;
    ctx->prod_alloc += bytes;
    if (ctx->cap) return graph_alloc_bytes(ctx, p, bytes);
    auto it = ctx->free_blocks.lower_bound(bytes);
    if (it != ctx->free_blocks.end() && it->first - bytes <= it->first / 4) {
        *p = it->second;
        size_t sz = it->first;
        ctx->live_blocks[*p] = sz;
        ctx->cached_bytes -= sz;
        ctx->free_blocks.erase(it);
        return poison(ctx, *p, sz);
    }
    if (ctx->cached_bytes > ctx->cache_limit) pem_cache_release(ctx);
    cudaError_t e = cudaMallocFromPoolAsync(p, bytes, ctx->pool, ctx->stream);
    if (e == cudaErrorMemoryAllocation) {   // give the cached blocks back and try once more
        (void)cudaGetLastError();
        pem_cache_release(ctx);
        e = cudaMallocFromPoolAsync(p, bytes, ctx->pool, ctx->stream);
    }
    if (e != cudaSuccess) return ctx->fail_cuda(e, "cudaMallocFromPoolAsync", __FILE__, __LINE__);
    ctx->live_blocks[*p] = bytes;
    ctx->pool_taken += bytes;
    ++ctx->pool_mallocs;
    return poison(ctx, *p, bytes);
}

void pem_free_bytes(pem_ctx* ctx, void* p)
{
    if (ctx->cap && ctx->cap->owned.count(p)) {     // stays in the arena (and in live_blocks)
        ctx->cap->idle.emplace(ctx->live_blocks[p], p);
        return;
    }
    auto it = ctx->live_blocks.find(p);
    if (it == ctx->live_blocks.end()) {     // not ours (should not happen): plain stream-ordered free
        cudaFreeAsync(p, ctx->stream);
        return;
    }
    ctx->free_blocks.emplace(it->second, p);
    ctx->cached_bytes += it->second;
    ctx->live_blocks.erase(it);
}

// a graph hands its arena back to the shared cache when the last holder (its plan, or a result borrowed from it) lets go
pem_graph::~pem_graph()
{
    if (exec) cudaGraphExecDestroy(exec);
    if (!ctx) return;
    for (auto& b : arena)
        if (ctx->live_blocks.count(b.first)) pem_free_bytes(ctx, b.first);
    ctx->graph_bytes -= std::min(ctx->graph_bytes, bytes);
}

void pem_graph_opts(const pem_ctx* ctx, int* o)
{
    o[0] = ctx->opt_owner; o[1] = ctx->opt_step2_kernel; o[2] = ctx->opt_s3_small_e; o[3] = ctx->opt_s3_small_np; o[4] = ctx->opt_trace;
}

void pem_cache_release(pem_ctx* ctx)
{
    for (auto& kv : ctx->free_blocks) {
        cudaFreeAsync(kv.second, ctx->stream);
        ctx->pool_taken -= std::min(ctx->pool_taken, kv.first);
    }
    ctx->free_blocks.clear();
    ctx->cached_bytes = 0;
    cudaStreamSynchronize(ctx->stream);
    cudaMemPoolTrimTo(ctx->pool, 0);
}

extern "C" {

int pem_ctx_create(pem_ctx** out, int device)
{
    if (!out) return PEM_ERR_ARG;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) {
        (void)cudaGetLastError();
        return PEM_ERR_NO_DEVICE;
    }
    pem_ctx* ctx = new (std::nothrow) pem_ctx();
    if (!ctx) return PEM_ERR_ARG;
    ctx->device = device;
    auto bail = [&](cudaError_t e) {
        fprintf(stderr, "pem_ctx_create: %s\n", cudaGetErrorString(e));
        delete ctx;
        return PEM_ERR_CUDA;
    };
    cudaError_t e;
    if ((e = cudaSetDevice(device)) != cudaSuccess) return bail(e);
    if ((e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess) return bail(e);
    if ((e = cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking)) != cudaSuccess) return bail(e);
    for (auto& ev : ctx->ev_copy)
        if ((e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming)) != cudaSuccess) return bail(e);
    cudaMemPoolProps props = {};
    props.allocType = cudaMemAllocationTypePinned;
    props.handleTypes = cudaMemHandleTypeNone;
    props.location.type = cudaMemLocationTypeDevice;
    props.location.id = device;
    if ((e = cudaMemPoolCreate(&ctx->pool, &props)) != cudaSuccess) return bail(e);
    uint64_t never = UINT64_MAX;
    if ((e = cudaMemPoolSetAttribute(ctx->pool, cudaMemPoolAttrReleaseThreshold, &never)) != cudaSuccess) return bail(e);
    if ((e = cudaMallocHost((void**)&ctx->h_scalars, PEM_NSCALARS * sizeof(int64_t))) != cudaSuccess) return bail(e);
    if ((e = cudaMallocHost((void**)&ctx->h_check, PEM_PLAN_MAX * sizeof(int64_t))) != cudaSuccess) return bail(e);
    if ((e = cudaMalloc((void**)&ctx->d_scalars, PEM_NSCALARS * sizeof(int64_t))) != cudaSuccess) return bail(e);
    for (auto& ev : ctx->ev)
        if ((e = cudaEventCreate(&ev)) != cudaSuccess) return bail(e);
    for (auto& ev : ctx->kev)
        if ((e = cudaEventCreate(&ev)) != cudaSuccess) return bail(e);
    cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device);
    cudaDeviceGetAttribute(&ctx->smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) {
        ctx->cache_limit = free_b / 5 * 4;      // of what was FREE at creation: other allocators in the process keep theirs
        ctx->graph_limit = free_b / 4;
        ctx->free_at_create = free_b;
    }
    *out = ctx;
    return PEM_OK;
}

void pem_ctx_destroy(pem_ctx* ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    ctx->plans.clear();                      // idle product graphs hand their arenas back to the cache
    pem_cache_release(ctx);
    for (auto& kv : ctx->live_blocks) cudaFreeAsync(kv.first, ctx->stream);   // handles the caller leaked
    cudaStreamSynchronize(ctx->stream);
    for (auto& ev : ctx->ev)
        if (ev) cudaEventDestroy(ev);
    for (auto& ev : ctx->kev)
        if (ev) cudaEventDestroy(ev);
    if (ctx->d_scalars) cudaFree(ctx->d_scalars);
    if (ctx->h_scalars) cudaFreeHost(ctx->h_scalars);
    if (ctx->h_check) cudaFreeHost(ctx->h_check);
    if (ctx->pool) cudaMemPoolDestroy(ctx->pool);
    for (auto& ev : ctx->ev_copy)
        if (ev) cudaEventDestroy(ev);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

const char* pem_last_error(const pem_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int pem_ctx_set_option(pem_ctx* ctx, int option, int64_t value)
{
    if (!ctx) return PEM_ERR_ARG;
    switch (option) {
        case PEM_OPT_KEEP_EMPTY_TILES: ctx->opt_keep_empty = value != 0; return PEM_OK;
        case PEM_OPT_STEP1_PATH:
            if (value < 0 || value > 5) return ctx->fail(PEM_ERR_ARG, "PEM_OPT_STEP1_PATH must be 0..5");
            ctx->opt_step1_path = (int)value;
            return PEM_OK;
        case PEM_OPT_OWNER:
            if (value < 0 || value > 4) return ctx->fail(PEM_ERR_ARG, "PEM_OPT_OWNER must be 0..4");
            ctx->opt_owner = (int)value;
            return PEM_OK;
        case PEM_OPT_TRACE: ctx->opt_trace = (int)value; return PEM_OK;
        case PEM_OPT_SIZE_PLANS:
            ctx->opt_plans = value != 0;
            ctx->plans.clear();
            return PEM_OK;
        case PEM_OPT_GRAPHS:
            ctx->opt_graphs = value != 0;
            for (auto& kv : ctx->plans) { kv.second.graph.reset(); kv.second.graph_failed = false; }
            return PEM_OK;
        case PEM_OPT_GRAPH_LIMIT_MB:
            if (value < 0) return ctx->fail(PEM_ERR_ARG, "PEM_OPT_GRAPH_LIMIT_MB must be >= 0");
            ctx->graph_limit = (size_t)value << 20;
            return PEM_OK;
        case PEM_OPT_ESC_VARIANT:
            if (value < 0 || value > 3) return ctx->fail(PEM_ERR_ARG, "PEM_OPT_ESC_VARIANT must be 0..3");
            ctx->opt_esc_variant = (int)value;
            return PEM_OK;
        case PEM_OPT_CACHE_LIMIT_MB:
            if (value < 0) return ctx->fail(PEM_ERR_ARG, "PEM_OPT_CACHE_LIMIT_MB must be >= 0");
            ctx->cache_limit = (size_t)value << 20;
            if (ctx->cached_bytes > ctx->cache_limit) pem_cache_release(ctx);
            return PEM_OK;
        case PEM_OPT_STEP2_KERNEL:
            if (value < 0 || value > 3) return ctx->fail(PEM_ERR_ARG, "PEM_OPT_STEP2_KERNEL must be 0..3");
            ctx->opt_step2_kernel = (int)value;
            return PEM_OK;
        case PEM_OPT_ASYNC_VALUES: ctx->opt_async_vals = value != 0; return PEM_OK;
        case PEM_OPT_S3_SMALL_NNZ:
            if (value < 0 || value > 256) return ctx->fail(PEM_ERR_ARG, "PEM_OPT_S3_SMALL_NNZ must be 0..256");
            ctx->opt_s3_small_e = (int)value;
            return PEM_OK;
        case PEM_OPT_S3_SMALL_PAIRS:
            if (value < 0 || value > (1 << 20)) return ctx->fail(PEM_ERR_ARG, "PEM_OPT_S3_SMALL_PAIRS must be 0..2^20");
            ctx->opt_s3_small_np = (int)value;
            return PEM_OK;
        case PEM_OPT_POISON:
            if (value != 0 && (value < 0x100 || value > 0x1FF))
                return ctx->fail(PEM_ERR_ARG, "PEM_OPT_POISON must be 0 or 0x100 | byte");
            ctx->opt_poison = (int)value;
            ctx->plans.clear();      // a graph captured without the fill nodes must not run again
            return PEM_OK;
    }
    return ctx->fail(PEM_ERR_ARG, "unknown option");
}

void* pem_ctx_stream(pem_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

int pem_ctx_sync(pem_ctx* ctx)
{
    if (!ctx) return PEM_ERR_ARG;
    PEM_CK(cudaStreamSynchronize(ctx->stream));
    return PEM_OK;
}

int64_t pem_ctx_launch_count(const pem_ctx* ctx) { return ctx ? ctx->launches : 0; }
int pem_ctx_last_sort_passes(const pem_ctx* ctx) { return ctx ? ctx->last_sort_passes : -1; }

int pem_ctx_kernel_ms(const pem_ctx* ctx, double* ms, int n)
{
    if (!ctx || !ms || n < KT_N) return PEM_ERR_ARG;
    for (int i = 0; i < KT_N; ++i) ms[i] = ctx->kt_ms[i];
    return KT_N;
}

int pem_ctx_last_step3_kernel(const pem_ctx* ctx) { return ctx ? ctx->last_step3_kernel : 0; }

int64_t pem_ctx_size_stalls(const pem_ctx* ctx) { return ctx ? ctx->size_stalls : 0; }

int64_t pem_ctx_pool_mallocs(const pem_ctx* ctx) { return ctx ? ctx->pool_mallocs : 0; }

int64_t pem_ctx_graph_replays(const pem_ctx* ctx) { return ctx ? ctx->graph_replays : 0; }

int pem_ctx_trim(pem_ctx* ctx)
{
    if (!ctx) return PEM_ERR_ARG;
    PEM_CK(cudaSetDevice(ctx->device));
    pem_cache_release(ctx);
    return PEM_OK;
}

int64_t pem_ctx_pool_bytes(const pem_ctx* ctx)
{
    if (!ctx) return 0;
    uint64_t v = 0;
    cudaMemPoolGetAttribute(ctx->pool, cudaMemPoolAttrReservedMemCurrent, &v);
    return (int64_t)v;
}

// ---- tiled accessors -----------------------------------------------------------------------
int pem_tiled_info_get(const pem_tiled* t, pem_tiled_info* info)
{
    if (!t || !info) return PEM_ERR_ARG;
    info->rows = t->rows; info->cols = t->cols; info->nnz = t->nnz;
    info->tile_rows = t->tile_rows; info->tile_cols = t->tile_cols; info->tiles = t->tiles;
    return PEM_OK;
}

static const void* tiled_array(const pem_tiled* t, int which, size_t* bytes)
{
    size_t n = (size_t)t->tiles;
    switch (which) {
        case PEM_T_VALS: *bytes = (size_t)t->nnz * pem_vsize(t->dtype); return t->vals;
        case PEM_T_TILE_NNZ_PTR: *bytes = (n + 1) * 4; return t->tile_nnz_ptr;
        case PEM_T_MASKS: *bytes = n * 32; return t->masks;
        case PEM_T_ROW_PTR: *bytes = n * 16; return t->row_ptr;
        case PEM_T_MASKS_T: *bytes = n * 32; return t->masks_t;
        case PEM_T_TILE_ROW_PTR: *bytes = ((size_t)t->tile_rows + 1) * 4; return t->tile_row_ptr;
        case PEM_T_TILE_COL_IDX: *bytes = n * 4; return t->tile_col_idx;
        case PEM_T_TILE_ROW_IDX: *bytes = n * 4; return t->tile_row_idx;
        case PEM_T_COL_OCC: *bytes = n * 2; return t->col_occ;
        case PEM_T_ROW_OCC: *bytes = n * 2; return t->row_occ;
        case PEM_T_ROW_COL_IDX: *bytes = (size_t)t->nnz; return t->rc_idx;
        case PEM_T_VAL_POS: *bytes = (size_t)t->nnz * 4; return t->val_pos;
    }
    *bytes = 0;
    return nullptr;
}

int pem_tiled_dtype(const pem_tiled* t) { return t ? t->dtype : -1; }
int pem_result_dtype(const pem_result* C) { return C ? C->dtype : -1; }

int pem_tiled_values_ready(pem_ctx* ctx, const pem_tiled* t)
{
    if (!ctx || !t) return PEM_ERR_ARG;
    if (t->vals_pending) PEM_CK(cudaEventSynchronize(t->ev_vals));
    return PEM_OK;
}

const void* pem_tiled_device_ptr(const pem_tiled* t, int which)
{
    size_t b;
    if (t && which == PEM_T_VALS && t->vals_pending) cudaEventSynchronize(t->ev_vals);   // no context here: wait on the host
    return t ? tiled_array(t, which, &b) : nullptr;
}

int pem_tiled_get(pem_ctx* ctx, const pem_tiled* t, int which, void* host_dst, size_t bytes)
{
    if (!ctx || !t || !host_dst) return PEM_ERR_ARG;
    size_t have = 0;
    const void* src = tiled_array(t, which, &have);
    if (!src && have == 0 && which > PEM_T_VAL_POS) return ctx->fail(PEM_ERR_ARG, "unknown tiled array");
    if (bytes != have) return ctx->fail(PEM_ERR_ARG, "pem_tiled_get: size mismatch");
    if (bytes == 0) return PEM_OK;
    if (which == PEM_T_VALS) PEM_TRY(pem_tiled_wait_vals(ctx, t));
    PEM_CK(cudaMemcpyAsync(host_dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    PEM_CK(cudaStreamSynchronize(ctx->stream));
    return PEM_OK;
}

void pem_tiled_free(pem_ctx* ctx, pem_tiled* t)
{
    if (!ctx || !t) return;
    (void)pem_tiled_wait_vals(ctx, t);       // a gather still in flight on the copy stream writes t->vals
    if (t->ev_vals) cudaEventDestroy(t->ev_vals);
    for (auto it = ctx->plans.begin(); it != ctx->plans.end();) {    // size plans and product graphs of this operand
        if ((uint64_t)it->first[0] == t->uid || (uint64_t)it->first[1] == t->uid) it = ctx->plans.erase(it);
        else ++it;
    }
    for (void** f : t->buffers()) pem_free(ctx, *f);
    delete t;
}

// ---- result accessors ----------------------------------------------------------------------
int pem_result_info_get(const pem_result* C, pem_result_info* info)
{
    if (!C || !info) return PEM_ERR_ARG;
    info->tile_row_begin = C->rb; info->tile_row_end = C->re;
    info->rows = C->rows; info->cols = C->cols;
    info->tiles = C->tiles; info->pairs = C->pairs; info->nnz = C->nnz;
    info->tile_products = C->tile_products;
    return PEM_OK;
}

static const void* result_array(const pem_result* C, int which, size_t* bytes)
{
    size_t n = (size_t)C->tiles;
    switch (which) {
        case PEM_R_ROW_PTR: *bytes = ((size_t)(C->re - C->rb) + 1) * 8; return C->row_ptr;
        case PEM_R_TILE_ROW: *bytes = n * 4; return C->tile_row;
        case PEM_R_TILE_COL: *bytes = n * 4; return C->tile_col;
        case PEM_R_PAIR_PTR: *bytes = (n + 1) * 8; return C->pair_ptr;
        case PEM_R_PAIRS_A: *bytes = (size_t)C->pairs * 4; return C->pair_list;                   // stride 8 bytes
        case PEM_R_PAIRS_B: *bytes = (size_t)C->pairs * 4; return (const int32_t*)C->pair_list + 1;   // stride 8 bytes
        case PEM_R_MASKS: *bytes = C->stage >= 2 ? n * 32 : 0; return C->masks;
        case PEM_R_TILE_NNZ_PTR: *bytes = C->stage >= 2 ? (n + 1) * 8 : 0; return C->tile_nnz_ptr;
        case PEM_R_ROW_COL_IDX: *bytes = C->stage >= 2 ? (size_t)C->nnz : 0; return C->row_col_idx;
        case PEM_R_VALS: *bytes = C->stage >= 3 ? (size_t)C->nnz * pem_vsize(C->dtype) : 0; return C->vals;
    }
    *bytes = 0;
    return nullptr;
}

const void* pem_result_device_ptr(const pem_result* C, int which)
{
    size_t b;
    return C ? result_array(C, which, &b) : nullptr;
}

int pem_result_get(pem_ctx* ctx, const pem_result* C, int which, void* host_dst, size_t bytes)
{
    if (!ctx || !C || !host_dst) return PEM_ERR_ARG;
    if (which == PEM_R_ROW_COL_IDX && C->stage >= 2) PEM_TRY(pem_result_make_rowcolidx(ctx, const_cast<pem_result*>(C)));
    size_t have = 0;
    const void* src = result_array(C, which, &have);
    if (bytes != have) return ctx->fail(PEM_ERR_ARG, "pem_result_get: size mismatch (or stage not run yet)");
    if (bytes == 0) return PEM_OK;
    if (which == PEM_R_PAIRS_A || which == PEM_R_PAIRS_B)   // stored interleaved as int2 on the device
        PEM_CK(cudaMemcpy2DAsync(host_dst, 4, src, 8, 4, (size_t)C->pairs, cudaMemcpyDeviceToHost, ctx->stream));
    else
        PEM_CK(cudaMemcpyAsync(host_dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    PEM_CK(cudaStreamSynchronize(ctx->stream));
    return PEM_OK;
}

void pem_result_free(pem_ctx* ctx, pem_result* C)
{
    if (!ctx || !C) return;
    if (C->graph) {
        // buffers borrowed from a product graph stay in its arena (the graph may run again now); anything added to
        // the result later (Ctiles_rowColIdx on demand) was allocated the ordinary way
        for (void** f : C->buffers())
            if (*f && C->graph->owned.count(*f)) *f = nullptr;
        C->graph->busy = false;
    }
    for (void** f : C->buffers()) pem_free(ctx, *f);
    delete C;
}

}  // extern "C"

// In-place exclusive prefix sum over n int64 values (CUB device scan as a building block; the
// reference uses thrust::exclusive_scan at the same places, spgemm.cu:1168,1242,1288).
int pem_scan_exclusive_i64(pem_ctx* ctx, int64_t* d, int64_t n)
{
    if (n <= 0) return PEM_OK;
    size_t tmp_bytes = 0;
    PEM_CK(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, d, d, n, ctx->stream));
    char* tmp = nullptr;
    pem_guard g(ctx, tmp);
    PEM_TRY(pem_alloc(ctx, &tmp, tmp_bytes));
    PEM_CK(cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, d, d, n, ctx->stream));
    pem_free(ctx, tmp);
    return PEM_OK;
}
