/*
 * pemspgemm.h — C ABI of the B200-native SpGEMM engine (libpemspgemm.so).
 *
 * The reference (stckvrflw/pem-spgemm, /root/reference) has no library, plugin or FFI
 * layer: conversion, the three SpGEMM steps, timing and the result dump are inline in
 * `main` (spgemm.cu:720-1568).  This header cuts that function at its stage boundaries so
 * that a host program (the `pemspgemm` CLI in this repo, the reference's own `main`, a
 * ctypes/cgo/JNI binding) can call the hot path as a drop-in.  Each entry point names the
 * region of the reference it replaces.
 *
 * Conventions: plain pointers and sizes only; every function returns PEM_OK (0) or a
 * negative pem_status and never calls exit(); `pem_last_error` gives the message.  A
 * context owns one CUDA stream and one stream-ordered memory pool (cudaMemPool_t) on one
 * device; it is not thread-safe; use one context per GPU.  Opaque handles own device
 * memory from the context's pool and must be freed through this ABI before the context.
 * There is no CPU fallback: without a CUDA device pem_ctx_create fails.
 */
#ifndef PEMSPGEMM_H
#define PEMSPGEMM_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PEM_TILE 16 /* tile edge, spgemm.cu:727 */

typedef enum pem_status {
    PEM_OK = 0,
    PEM_ERR_CUDA = -1,       /* a CUDA runtime call failed (message has the call site)      */
    PEM_ERR_ARG = -2,        /* bad argument (null handle, negative size, shape mismatch)   */
    PEM_ERR_RANGE = -3,      /* a COO coordinate is outside rows x cols                     */
    PEM_ERR_DUPLICATE = -4,  /* the COO input holds the same (i,j) twice (reference: UB)    */
    PEM_ERR_LIMIT = -5,      /* a size exceeds what the engine supports (see message)       */
    PEM_ERR_NO_DEVICE = -6,  /* no usable CUDA device                                       */
    PEM_ERR_IO = -7          /* file could not be read / parsed / written                   */
} pem_status;

typedef struct pem_ctx pem_ctx;       /* stream + memory pool + scratch, one per GPU */
typedef struct pem_tiled pem_tiled;   /* a matrix in 16x16 tiled-CSR form (SURVEY.md 2.2) */
typedef struct pem_result pem_result; /* C (or a tile-row panel of C) in tiled form */

/* Engine options (pem_ctx_set_option). */
typedef enum pem_option {
    /* 0 (default): step 1 drops (A tile, B tile) pairs whose 16x16 boolean product is empty, so
     *    C' holds exactly the non-empty tiles of C.
     * 1: reference-faithful C': every structurally reachable tile and pair is kept, including
     *    empty ones (spgemm.cu:271-384 works on the tile structure only; "C tiles" in the
     *    reference's report counts them, spgemm.cu:1420).  C itself is identical either way. */
    PEM_OPT_KEEP_EMPTY_TILES = 1,
    /* step-1 algorithm: 0 (default) = automatic: expand-sort-compress over tile products (no
     * per-row accumulator, no limit on tile columns), except for small operands (<= 64K tiles and a
     * tile-column window that fits shared memory) where the per-row bitmap path has fewer launches;
     * 1 = force the per-row windowed bitmap accumulator (the reference's SPA idea,
     * spgemm.cu:271-384); 2 = force expand-sort-compress; 3 / 4 = expand-sort-compress with the
     * tile-level / row-sliced product expansion forced (2 picks the one with fewer products); 5 = the per-row path with
     * HASH accumulators (open addressing in shared memory, the NSPARSE idea) on every tile row of at most 1024 tile
     * products and the bitmap on the others (1 / automatic use the hash only on rows whose window of tile columns is
     * more than 16 x wider than their products).  Replaces the reference's global switch between
     * SPA and NSPARSE hashing `B_tileCols > 512*32` (spgemm.cu:1142). */
    PEM_OPT_STEP1_PATH = 2,
    /* thread mapping of step 3 (and of step 2 for value 1).  Results are bit-identical.
     * 0 (default) = automatic: the window kernel (4) when C holds at least four nonzeros per tile pair (stencil /
     *     FEM products), else the entry-owner kernel (2)
     * 2 = entry-owner: one thread per C nonzero over the flat nonzero index space
     * 1 = row-owner: sixteen lanes per C' tile, lane = tile row (steps 2 and 3; no pair kernel)
     * 3 = tile-class kernel: a warp takes 32 consecutive C' tiles; small tiles get one thread each, the
     *     others one warp each with their pairs' records staged in shared memory (or, for long pair
     *     lists, found through step 2's hit blocks)
     * 4 = window kernel: a block takes the C' tiles of a 128-pair window of the pair list, stages the pairs' A row
     *     records / B column records in shared memory (128-bit asynchronous copies), decodes the window's nonzeros
     *     cooperatively and lets each thread own nonzeros */
    PEM_OPT_OWNER = 3,
    /* tuning of the tile-class kernel: a C' tile with at most SMALL_NNZ nonzeros (default 8) and at most
     * SMALL_PAIRS pairs (default 64) is handled by one thread, any other tile by one warp */
    PEM_OPT_S3_SMALL_NNZ = 4,
    PEM_OPT_S3_SMALL_PAIRS = 5,
    /* 0 (default): when pem_convert_coo returns, the caller's I/J/V arrays are free again.
     * 1: for HOST input, pem_convert_coo returns while the upload of V (half of the COO bytes) is still in
     *    flight on the context's copy stream; V must stay valid and unmodified until pem_tiled_values_ready
     *    (or any product / accessor that reads the values) has returned.  The symbolic steps 1 and 2 of a
     *    product read masks only, so they overlap the upload: on config 4 end to end 51 -> 45 ms. */
    PEM_OPT_ASYNC_VALUES = 6,
    /* step-2 mask kernel: one lane per (A tile, B tile) pair, 1 = walking the shorter nonzero list, 3 = from the
     * two tiles' row masks alone (128-bit mask loads, product rows in registers), 0 (default) = 3 when A's tiles
     * hold at least eight nonzeros on average, else 1; 2 = sixteen lanes per C' tile, row masks exchanged by
     * shuffles (bit-identical; measured slower) */
    PEM_OPT_STEP2_KERNEL = 7,
    /* diagnostics: 1 = host-side timeline of step 1 on stderr (where the host waits), 2 = also per-phase cycle
     * counters of the bitmap kernels */
    PEM_OPT_TRACE = 8,
    /* expand-sort-compress variants that are otherwise chosen by size (tests force them): bit 0 = count per chunk,
     * scan, write exactly (instead of staging at product bases and compacting), bit 1 = never use the block-local
     * row sort */
    PEM_OPT_ESC_VARIANT = 9,
    /* the context keeps freed device blocks for reuse; once more than this many MiB are cached they are handed
     * back to the driver (default: 80 % of the memory free at pem_ctx_create); see pem_ctx_trim */
    PEM_OPT_CACHE_LIMIT_MB = 10,
    /* 1 (default): pem_spgemm / pem_spgemm_panel remember the sizes a product read back from the device (tile products,
     * kept pairs, C' tiles, nnz; spgemm.cu:1169, 1246, 1291 are the reference's three such stalls) per (A, B, panel)
     * and a repeated product of the same handles replays them: buffers are sized and grids launched from the
     * remembered values while every kernel still computes the sizes on the device, which are compared after the
     * product's single final synchronisation (on a mismatch the product is redone with the stalls).  0: every product
     * stalls at its read-backs (five per product).  Setting the option clears the remembered sizes. */
    PEM_OPT_SIZE_PLANS = 11,
    /* 1 (default): a repeated product whose sizes are remembered (PEM_OPT_SIZE_PLANS) is captured as ONE CUDA graph
     * the second time it runs and launched as such from then on: its ~20-40 kernels, memsets and size copies cost one
     * launch, which is what bounds small operands (config 1: 15 kernels for 0.15 ms of device time) and the short
     * per-GPU panels of a multi-GPU run.  The graph owns the device blocks its product touches, result included: a
     * result handed out from it borrows them, and the graph runs again only after that result was freed (a product
     * called while the previous result is alive takes the ordinary path).  A product with a host stall inside, or
     * whose blocks do not fit the graphs' memory budget (PEM_OPT_GRAPH_LIMIT_MB), silently stays on the ordinary path.
     * Freeing an operand drops its plans and graphs.  0: no graphs. */
    PEM_OPT_GRAPHS = 12,
    /* budget for the device memory held by product graphs, MiB (default: a quarter of the memory free at pem_ctx_create);
     * a single graph may hold an eighth of it: products that move gigabytes do not wait for their launches, and the
     * sequential panels of a large product must not park their buffers in graphs */
    PEM_OPT_GRAPH_LIMIT_MB = 13,
    /* tests only: 0 (default) = off; 0x100 | b (0 <= b <= 255) = every device block the context's allocator hands
     * out (a cached block in full, a new pool block, a block of a product graph's arena) is filled with byte b on the
     * context's stream before use, so a kernel that reads memory nothing wrote sees b, not the block's previous
     * contents or fresh zeros.  Inside a graph capture the fill becomes a node of the graph.  Not filled: the
     * context's scalar slots, pinned host memory and caller buffers.  Costs no kernel launch (memsets only).
     * Setting the option clears the remembered sizes and graphs, as PEM_OPT_SIZE_PLANS does. */
    PEM_OPT_POISON = 14
} pem_option;

/* Milliseconds.  Device times are CUDA-event times on the context's stream; wall times are
 * host clocks around the call with the stream drained on both sides (the reference's
 * pem_spgemm_time, spgemm.cu:1136,1340). */
typedef struct pem_times {
    double convert_kernel_ms; /* tile build kernel only  == A/B_conversion_kernel_time (spgemm.cu:938-978) */
    double convert_total_ms;  /* whole COO->tiled conversion incl. H2D copies (wall)                       */
    double step1_ms;          /* tile-level symbolic  == step1_time (spgemm.cu:1141-1218)                  */
    double step2_ms;          /* mask symbolic        == step2_time (spgemm.cu:1344-1350)                  */
    double step3_ms;          /* numeric              == step3_time (spgemm.cu:1348)                       */
    double kernel_ms;         /* step1+step2+step3    == pem_spgemm_kernel_time (spgemm.cu:1353)           */
    double total_ms;          /* wall for the call    == pem_spgemm_time (spgemm.cu:1352)                  */
    double malloc_ms;         /* total - kernel       == pem_spgemm_malloc_time (spgemm.cu:1354)           */
} pem_times;

typedef struct pem_tiled_info {
    int32_t rows, cols;           /* after the optional transpose */
    int64_t nnz;
    int32_t tile_rows, tile_cols; /* ceil(rows/16), ceil(cols/16), spgemm.cu:840-843 */
    int32_t tiles;                /* non-empty tiles (cntA / cntB, spgemm.cu:871,885) */
} pem_tiled_info;

typedef struct pem_result_info {
    int32_t tile_row_begin, tile_row_end; /* the panel of A' tile rows this result covers */
    int32_t rows, cols;                   /* shape of the full C */
    int64_t tiles;                        /* C' tiles        ("C tiles",  spgemm.cu:1420) */
    int64_t pairs;                        /* (A tile,B tile) pairs (d_pairs_count, spgemm.cu:1246) */
    int64_t nnz;                          /* nnz of C         ("C nnz",   spgemm.cu:1421) */
    int64_t tile_products;                /* tile-level intermediate products examined by step 1 */
} pem_result_info;

/* ---- context ------------------------------------------------------------------------ */
/* Replaces the stream / RMM pool setup at spgemm.cu:757-758,808-817. */
int pem_ctx_create(pem_ctx** out, int device);
void pem_ctx_destroy(pem_ctx* ctx);
const char* pem_last_error(const pem_ctx* ctx); /* valid until the next call on ctx */
int pem_ctx_set_option(pem_ctx* ctx, int option, int64_t value);
void* pem_ctx_stream(pem_ctx* ctx);             /* the cudaStream_t all work is enqueued on */
int pem_ctx_sync(pem_ctx* ctx);
/* Number of kernels this library launched on ctx since creation (bench.py's gpu_launches). */
int64_t pem_ctx_launch_count(const pem_ctx* ctx);
/* Device time (ms, CUDA events on the context's stream) of the four individually timed kernels of
 * the last pem_spgemm / pem_spgemm_panel call (pem_spgemm_numeric: [3] only, the others 0): [0] k_expand (step 1 product expansion), [1] the
 * step-1 radix sort, [2] k_step2_pairs, [3] the step-3 numeric kernel.  Returns the count (4). */
int pem_ctx_kernel_ms(const pem_ctx* ctx, double* ms, int n);
/* How step 1 of the last product ordered its tile pairs: -1 = no sort (per-row bitmap path), 0 = block-local
 * sort of every C' row in shared memory, n > 0 = n passes of the global radix sort (labels the KT slot [1]). */
int pem_ctx_last_sort_passes(const pem_ctx* ctx);
/* Which numeric kernel step 3 of the last product ran (PEM_OPT_OWNER 0 chooses): 1 = row-owner, 2 = entry-owner,
 * 3 = tile-class, 4 = window kernel (labels the KT slot [3] of pem_ctx_kernel_ms). */
int pem_ctx_last_step3_kernel(const pem_ctx* ctx);
/* Host stalls at device-size read-backs inside products since creation (diagnostic: five per first product of an
 * operand pair, none for its repeats under PEM_OPT_SIZE_PLANS; every product ends with one synchronisation). */
int64_t pem_ctx_size_stalls(const pem_ctx* ctx);
/* Products that ran as a single graph launch since creation (PEM_OPT_GRAPHS; diagnostic). */
int64_t pem_ctx_graph_replays(const pem_ctx* ctx);
/* Allocations that missed the context's block cache and went to the CUDA pool since creation
 * (diagnostic: a steady-state loop should not add any). */
int64_t pem_ctx_pool_mallocs(const pem_ctx* ctx);
/* Bytes currently reserved by the context's pool (diagnostic). */
int64_t pem_ctx_pool_bytes(const pem_ctx* ctx);
/* Hands every cached (freed, not yet reused) device block back to the driver: call between workloads when
 * another allocator in the process (torch, NCCL) needs the memory.  Synchronises the context's stream. */
int pem_ctx_trim(pem_ctx* ctx);

/* ---- conversion: COO -> tiled CSR ----------------------------------------------------- */
/* Replaces spgemm.cu:821-1066 (decide_which_tile, the thrust sort/unique/reduce pipeline,
 * generate_tiles_csr, __transpose_B_mask, tile-level CSR build).  I/J/V may be host or device
 * pointers (0-based, any order, no duplicates).  transpose != 0 converts the transposed matrix
 * (the CLI's B = A^T mode, spgemm.cu:788-792).  times may be NULL. */
int pem_convert_coo(pem_ctx* ctx, int32_t rows, int32_t cols, int64_t nnz,
                    const int32_t* I, const int32_t* J, const double* V, int transpose,
                    pem_tiled** out, pem_times* times);
/* The fp32 instantiation (the reference's kernels are templates over ValueType, spgemm.cu:137,593,727-728, and
 * ship as double only): same conversion with float values.  A product of two fp32 operands accumulates with
 * single-precision fma in the same ascending-k order and yields an fp32 result (pem_result_to_coo_f32;
 * pem_result_get(PEM_R_VALS) and pem_tiled_get(PEM_T_VALS) then move 4-byte values).  Operands of different
 * value types cannot be multiplied.  fp32 runs the default kernels (PEM_OPT_OWNER 0 / 2 / 4). */
int pem_convert_coo_f32(pem_ctx* ctx, int32_t rows, int32_t cols, int64_t nnz,
                        const int32_t* I, const int32_t* J, const float* V, int transpose,
                        pem_tiled** out, pem_times* times);
/* 0 = fp64, 1 = fp32 */
int pem_tiled_dtype(const pem_tiled* t);
int pem_result_dtype(const pem_result* C);
/* Same from CSR (the reference builds a CSR on its way to tiles, spgemm.cu:894-928; SURVEY.md section 8f rank 4
 * asks for a CSR-in entry): row_ptr[rows+1] (int32, starts at 0), col_idx / vals [row_ptr[rows]], all three host or
 * all three device pointers; columns need not be sorted inside a row; duplicates are rejected. */
int pem_convert_csr(pem_ctx* ctx, int32_t rows, int32_t cols, const int32_t* row_ptr, const int32_t* col_idx,
                    const double* vals, int transpose, pem_tiled** out, pem_times* times);
/* The transpose of a tiled matrix, built on the device from A's tiles (tile keys re-sorted, masks and
 * column masks swap roles, values moved to their column-major slots): B = A^T for the CLI's
 * `[1]` mode without parsing, uploading and sorting the COO a second time (the reference converts
 * the file twice, spgemm.cu:778-792, 849-978).  Bit-identical to pem_convert_coo(..., transpose=1). */
int pem_tiled_transpose(pem_ctx* ctx, const pem_tiled* A, pem_tiled** out);
/* Blocks the host until the values of a tiled matrix converted under PEM_OPT_ASYNC_VALUES have left the
 * caller's V array (immediate otherwise). */
int pem_tiled_values_ready(pem_ctx* ctx, const pem_tiled* t);
int pem_tiled_info_get(const pem_tiled* t, pem_tiled_info* info);
void pem_tiled_free(pem_ctx* ctx, pem_tiled* t);

/* Arrays of a tiled matrix (SURVEY.md 2.2), copied to host for tests / interop. */
typedef enum pem_tiled_array {
    PEM_T_VALS = 0,         /* double  [nnz]      *tiles_vals      */
    PEM_T_TILE_NNZ_PTR = 1, /* uint32  [tiles+1]  *_perTileNnz     */
    PEM_T_MASKS = 2,        /* uint16  [tiles*16] *tiles_masks     */
    PEM_T_ROW_PTR = 3,      /* uint8   [tiles*16] *tiles_rowPtr    */
    PEM_T_MASKS_T = 4,      /* uint16  [tiles*16] Btiles_transposed_mask */
    PEM_T_TILE_ROW_PTR = 5, /* int32   [tile_rows+1] _X_tileRowPtr */
    PEM_T_TILE_COL_IDX = 6, /* int32   [tiles]    _X_tileColIdx    */
    PEM_T_TILE_ROW_IDX = 7, /* int32   [tiles]    tile row of each tile */
    PEM_T_COL_OCC = 8,      /* uint16  [tiles]    OR of the tile's row masks    */
    PEM_T_ROW_OCC = 9,      /* uint16  [tiles]    OR of the tile's column masks */
    PEM_T_ROW_COL_IDX = 10, /* uint8   [nnz]      *tiles_rowColIdx: (r<<4)|c per value (spgemm.cu:195,221) */
    PEM_T_VAL_POS = 11      /* uint32  [nnz]      index of each value in the COO / CSR arrays the matrix was converted
                             *                    from (for a pem_tiled_transpose result: its source's input), the
                             *                    order pem_tiled_set_values reads V in */
} pem_tiled_array;
int pem_tiled_get(pem_ctx* ctx, const pem_tiled* t, int which, void* host_dst, size_t bytes);
/* Device pointer of the same arrays (no copy; owned by the handle). */
const void* pem_tiled_device_ptr(const pem_tiled* t, int which);

/* ---- new values on the same pattern ----------------------------------------------------- */
/* New values for a tiled matrix whose pattern stays: V[nnz] in the order of the COO / CSR arrays the handle was
 * converted from (for a pem_tiled_transpose result: the order of its source's input, so one V refreshes A and A^T).
 * Host or device pointer.  Values are written in place: device pointers of the handle, size plans and product graphs
 * stay valid, and every later product reads the new values.  Results computed earlier keep theirs (see
 * pem_spgemm_numeric).  A host V is free again when the call returns.  A device V is read in the order of the
 * context's stream (pem_ctx_stream) without a host wait: the caller orders its own writes to V before this call and
 * after it on that stream.  A handle converted under PEM_OPT_ASYNC_VALUES first waits for its pending upload.  The
 * fp64 entry refuses an fp32 matrix and the reverse (PEM_ERR_ARG); nnz == 0 is a no-op. */
int pem_tiled_set_values(pem_ctx* ctx, pem_tiled* t, const double* V);
int pem_tiled_set_values_f32(pem_ctx* ctx, pem_tiled* t, const float* V);

/* ---- flop count and panel partition ---------------------------------------------------- */
/* flop = sum over a_ik of nnz(B row k); replaces the host thread at spgemm.cu:1068-1079. */
int pem_count_flop(pem_ctx* ctx, const pem_tiled* A, const pem_tiled* B, uint64_t* flop);
/* Split A's tile rows into nparts contiguous panels of balanced work (per-tile-row flop + 16 x the
 * tile products step 1 expands for the row, both counted on the device): bounds[0]=0,
 * bounds[nparts]=tile_rows (north_star: row-block tile-row panels by per-row flop count). */
int pem_partition_panels(pem_ctx* ctx, const pem_tiled* A, const pem_tiled* B, int nparts,
                         int32_t* bounds /* nparts+1 */);

/* ---- SpGEMM --------------------------------------------------------------------------- */
/* C = A*B: steps 1-3 with allocation, i.e. one iteration of the loop at spgemm.cu:1133-1357. */
int pem_spgemm(pem_ctx* ctx, const pem_tiled* A, const pem_tiled* B, pem_result** C, pem_times* times);
/* Same for the panel of A' tile rows [tile_row_begin, tile_row_end) (multi-GPU shards). */
int pem_spgemm_panel(pem_ctx* ctx, const pem_tiled* A, const pem_tiled* B,
                     int32_t tile_row_begin, int32_t tile_row_end, pem_result** C, pem_times* times);
/* Stage-level entry points (tests, ncu).  step1 creates the result handle; each later stage
 * requires the previous one.
 *   step1 : C' structure + ordered (A tile,B tile) pair lists
 *           (spgemm.cu:271-384 / NSPARSE hash path + pem_spgemm_step2_search_pairs, :387-497)
 *   step2 : C tile masks, per-tile nnz, scan, rowColIdx
 *           (pem_spgemm_step2_compute_CMasksAndOffsets :499-550, ..._CrowColIdx :552-591)
 *   step3 : values (pem_spgemm_step3_accumulate :593-661)                                  */
int pem_step1_symbolic(pem_ctx* ctx, const pem_tiled* A, const pem_tiled* B,
                       int32_t tile_row_begin, int32_t tile_row_end, pem_result** C);
int pem_step2_symbolic(pem_ctx* ctx, const pem_tiled* A, const pem_tiled* B, pem_result* C);
int pem_step3_numeric(pem_ctx* ctx, const pem_tiled* A, const pem_tiled* B, pem_result* C);

/* Recomputes the values of a complete result C of A*B (or of a panel of it) in place from the current values of
 * A and B, on C's existing structure: step 3 only, same kernel as C's first computation, no allocation of C's
 * buffers, no size read-back.  Bit-identical to a new pem_spgemm_panel of the same operands and panel.
 * A and B must be the handles C was computed from (A == B for A^2); PEM_ERR_ARG otherwise, and for a result that
 * has not completed step 3.  Works on a result handed out by a product graph.  Ends with one synchronisation;
 * times (may be NULL) gets step3_ms, kernel_ms, total_ms and malloc_ms, with steps 1 and 2 at 0. */
int pem_spgemm_numeric(pem_ctx* ctx, const pem_tiled* A, const pem_tiled* B, pem_result* C, pem_times* times);

/* ---- results as operands ---------------------------------------------------------------- */
/* A complete result C (or panel of C) as a new, independent tiled matrix: the next product of a chain (AMG's
 * P^T*(A*P), matrix powers, Markov clustering) without exporting C and converting it again.  Every array and
 * pem_tiled_info are identical to what pem_convert_coo builds from pem_result_to_coo(C)'s output (same dtype), so
 * the value map (PEM_T_VAL_POS) is the position of each value in C's sorted COO / CSR order, the order
 * pem_tiled_set_values then takes.  Empty C' tiles (PEM_OPT_KEEP_EMPTY_TILES) are dropped; explicit zeros of C stay.
 * A panel [tile_row_begin, tile_row_end) becomes a matrix of C's full shape whose tile rows outside the panel are
 * empty, so a panel product of it is the panel of the chained product.  The handle shares no memory with C: C may
 * be freed right after the call (a result borrowed from a product graph too, whose graph may then run again).  It
 * has an identity of its own for size plans and graphs.  PEM_ERR_ARG for a result before step 3, PEM_ERR_LIMIT for
 * nnz >= 2^32-1 or 2^31-1 tiles and more (as pem_convert_coo), both before anything is allocated.  Ends with one
 * synchronisation; a result made under PEM_OPT_KEEP_EMPTY_TILES = 1 adds one size read-back. */
int pem_result_to_tiled(pem_ctx* ctx, const pem_result* C, pem_tiled** out);
/* Writes the current values of C into a matrix t built by pem_result_to_tiled, in place, e.g. after
 * pem_spgemm_numeric recomputed C.  C must be a complete result of the same product and panel as the one t was
 * built from (the same A and B handles: C's structure depends on these alone), e.g. a later result of that product
 * handed out by its graph; PEM_ERR_ARG otherwise, and for a matrix not built by pem_result_to_tiled (a converted one,
 * or the pem_tiled_transpose of a built one: refresh those with pem_tiled_set_values).  As with pem_tiled_set_values,
 * device pointers of t (its values and, if built, their column-major view), size plans and product graphs stay
 * valid.  Stream-ordered on the context's stream: no allocation, no host wait. */
int pem_tiled_refresh_from_result(pem_ctx* ctx, pem_tiled* t, const pem_result* C);

/* ---- sums ------------------------------------------------------------------------------- */
/* S = alpha*A + beta*B as a new, independent tiled matrix (smoothed-aggregation prolongators P0 - w*(D^-1 A)*P0,
 * shifted operators A - s*I, A + A^T, graph Laplacians D - A), built on the device from the operands' tiles.
 *   Pattern: the union of the patterns of A and B.  Nothing is dropped: entries that cancel stay as explicit zeros,
 *     alpha = 0 or beta = 0 keeps the entries too, and explicit zeros of the operands stay.
 *   Values, exactly: an entry of both operands is fl(fl(alpha*a) + fl(beta*b)); an entry of A only is fl(alpha*a), one
 *     of B only fl(beta*b).  An absent entry is not a zero, so -0 and 0*Inf = NaN come out as IEEE says.  There is no
 *     fused multiply-add (e.g. alpha = 0.1, a = 10, beta = -1, b = 1 gives +0.0, where a fused form gives 2^-54 in
 *     fp64 and 2^-26 in fp32).  For fp32 operands alpha and beta are first rounded to float.
 *   The handle: every array and pem_tiled_info are identical to what pem_convert_coo builds from S's COO sorted by
 *     (row, col), in the operands' dtype; so the value map (PEM_T_VAL_POS) is each value's position in S's row-major
 *     order, the order pem_tiled_set_values then takes.  S shares no memory with A or B, which may be freed right after
 *     the call, and has an identity of its own for size plans and graphs.
 *   Operands: A and B may be the same handle, a pem_tiled_transpose, a pem_result_to_tiled handle or another sum.  An
 *     operand whose values are still uploading (PEM_OPT_ASYNC_VALUES) is waited for.
 *   Refusals: PEM_ERR_ARG for null handles, different shapes or different dtypes, before anything is allocated;
 *     PEM_ERR_LIMIT when the union holds 2^32-1 nonzeros or 2^31-1 tiles or more (as pem_convert_coo), after the size
 *     read-back, with nothing left allocated.
 *   Host waits: two size read-backs (the union's tiles, then its nnz) and one final synchronisation; a setup call, like
 *     a conversion. */
int pem_tiled_add(pem_ctx* ctx, double alpha, const pem_tiled* A, double beta, const pem_tiled* B, pem_tiled** out);
/* Rewrites the values of a sum S in place from the current values of A and B, with alpha and beta that may differ
 * from the build's: bit-identical to a new pem_tiled_add of the same values.  S must have been built by pem_tiled_add
 * from these two handles in this order; PEM_ERR_ARG otherwise: swapped operands, other handles, a matrix not built by
 * pem_tiled_add (a converted or pem_result_to_tiled one) and the pem_tiled_transpose of a sum.  S's device pointers
 * (its values and, if built, their column-major view), size plans and product graphs that read S stay valid.  No
 * allocation, no host wait: stream-ordered on the context's stream, after any pending upload of A or B. */
int pem_tiled_add_values(pem_ctx* ctx, pem_tiled* S, double alpha, const pem_tiled* A, double beta, const pem_tiled* B);

int pem_result_info_get(const pem_result* C, pem_result_info* info);
void pem_result_free(pem_ctx* ctx, pem_result* C);

typedef enum pem_result_array {
    PEM_R_ROW_PTR = 0,      /* int64  [panel tile rows+1]  _C_rowPtr            */
    PEM_R_TILE_ROW = 1,     /* int32  [tiles]              _C_tileRowIdx        */
    PEM_R_TILE_COL = 2,     /* int32  [tiles]              _C_tileColIdx        */
    PEM_R_PAIR_PTR = 3,     /* int64  [tiles+1]            pairs_insertion_offset */
    PEM_R_PAIRS_A = 4,      /* int32  [pairs]              d_pairs_a            */
    PEM_R_PAIRS_B = 5,      /* int32  [pairs]              d_pairs_b            */
    PEM_R_MASKS = 6,        /* uint16 [tiles*16]           Ctiles_mask (row r at index t*16+r) */
    PEM_R_TILE_NNZ_PTR = 7, /* int64  [tiles+1]            _C_perTileNnz        */
    PEM_R_ROW_COL_IDX = 8,  /* uint8  [nnz]                Ctiles_rowColIdx     */
    PEM_R_VALS = 9          /* double [nnz]                Ctiles_vals          */
} pem_result_array;
int pem_result_get(pem_ctx* ctx, const pem_result* C, int which, void* host_dst, size_t bytes);
const void* pem_result_device_ptr(const pem_result* C, int which);

/* Tiled C -> COO sorted by (row, col): sanitize_C + stable_sort + D2H (spgemm.cu:1493-1543).
 * rows/cols/vals are HOST buffers of pem_result_info.nnz entries (any may be NULL to skip). */
int pem_result_to_coo(pem_ctx* ctx, const pem_result* C, int32_t* rows, int32_t* cols, double* vals);
int pem_result_to_coo_f32(pem_ctx* ctx, const pem_result* C, int32_t* rows, int32_t* cols, float* vals);
/* Tiled C -> CSR with ascending columns: row_ptr is a HOST buffer of (rows covered by the result) + 1 int64 entries
 * (the whole C: rows + 1), cols / vals HOST buffers of nnz entries (any may be NULL to skip). */
int pem_result_to_csr(pem_ctx* ctx, const pem_result* C, int64_t* row_ptr, int32_t* cols, double* vals);
/* Same, but into DEVICE buffers, plus CSR row pointer (int64[rows_in_panel*16+1], may be NULL). */
int pem_result_to_coo_device(pem_ctx* ctx, const pem_result* C, int32_t* d_rows, int32_t* d_cols,
                             double* d_vals, int64_t* d_row_ptr);
/* Sum and sum of absolute values of C's values, reduced on the device (cheap result read-back
 * for end-to-end timing and smoke tests). */
int pem_result_checksum(pem_ctx* ctx, const pem_result* C, double* sum, double* abs_sum);

/* ---- Matrix Market I/O (host side; replaces fast_matrix_market use at spgemm.cu:43-110) ---- */
/* Reads coordinate real/integer/pattern/complex(real part) general/symmetric files into
 * malloc'ed arrays (free with pem_free_host).  Symmetric files are expanded. */
int pem_mtx_read(const char* path, int32_t* rows, int32_t* cols, int64_t* nnz,
                 int32_t** I, int32_t** J, double** V, int* is_symmetric, char* err, size_t err_len);
int pem_mtx_write(const char* path, int32_t rows, int32_t cols, int64_t nnz,
                  const int32_t* I, const int32_t* J, const double* V);
void pem_free_host(void* p);
/* One number per line, formatted on all host threads: the ROWS / COLS / VALS files of the reference's COO dump
 * (spgemm.cu:1545-1560, one `<<` per line there).  Doubles in fixed notation with 17 decimals, the digits
 * `std::fixed << std::setprecision(max_digits10)` prints (:1529).  append != 0 continues an existing file
 * (a result dumped panel by panel); otherwise the file is created or truncated. */
int pem_write_lines_i32(const char* path, const int32_t* x, int64_t n, int append);
int pem_write_lines_f64(const char* path, const double* x, int64_t n, int append);

#ifdef __cplusplus
}
#endif
#endif /* PEMSPGEMM_H */
