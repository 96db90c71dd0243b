// Sums of tiled matrices: S = alpha*A + beta*B as a new tiled operand, and its values recomputed in place.
//
// Both operands hold their tiles ordered by (tile row, tile column), and S's pattern is the union of theirs, so S's tile
// list is a merge of two sorted lists, done by ranks instead of a sort: every A tile finds its key in B's tile row by a
// binary search (whether B holds it, and how many B tiles come before it), every B tile does the same in A's; one scan
// over B's "not in A" flags then places every tile of the union.  The union gets the shape of a result (int64 tile-row
// pointer, tile rows and columns, row masks = the OR of the operands', int64 value offsets) and goes through the code
// pem_result_to_tiled runs (pem_operand_structure).  S keeps, per tile, the tile of A and of B it came from; from these
// k_add_vals computes every value, at the build and at every pem_tiled_add_values.  All of it is parallel over tiles or
// value slots, none of it over tile rows (power-law tile rows would serialise it).
#include "engine.cuh"

namespace {

// One thread per tile of A (g < na) and of B (the others): the lower bound of the tile's key in the other operand's
// tile row.  A tile i: a_rank[i] = that position in B if B holds the key, else its complement (negative).  B tile j:
// b_rank[j] = the position in A, b_new[j] = 1 when A does not hold the key.  Thread na + nb writes b_new[nb] = 0.
__global__ void __launch_bounds__(256)
k_sum_rank(int na, int nb, const int32_t* __restrict__ a_row, const int32_t* __restrict__ a_col,
           const int32_t* __restrict__ a_rp, const int32_t* __restrict__ b_row, const int32_t* __restrict__ b_col,
           const int32_t* __restrict__ b_rp, int32_t* __restrict__ a_rank, int32_t* __restrict__ b_rank,
           int64_t* __restrict__ b_new)
{
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t n = (int64_t)na + nb;
    if (g == n) b_new[nb] = 0;
    if (g >= n) return;
    const bool is_a = g < na;
    const int i = (int)(is_a ? g : g - na);
    const int r = (is_a ? a_row : b_row)[i], c = (is_a ? a_col : b_col)[i];
    const int32_t* rp = is_a ? b_rp : a_rp;
    const int32_t* col = is_a ? b_col : a_col;
    int lo = rp[r];
    const int end = rp[r + 1];
    int hi = end;
    while (lo < hi) {
        const int mid = lo + ((hi - lo) >> 1);
        if (col[mid] < c) lo = mid + 1; else hi = mid;
    }
    const bool hit = lo < end && col[lo] == c;
    if (is_a) {
        a_rank[i] = hit ? lo : ~lo;
    } else {
        b_rank[i] = lo;
        b_new[i] = hit ? 0 : 1;
    }
}

// One thread per tile of A and of B (u = exclusive scan of b_new): A tile i goes to i + u[rank of i in B], a B tile j
// that A does not hold to (rank of j in A) + u[j].  The thread writes the union tile's sources, key, OR of the row masks
// and its count of values (cnt[pos], scanned into the value offsets; thread na + nb writes cnt[ns] = 0).  Threads up to
// tile_rows write the union's tile-row pointer: A's tiles of the earlier tile rows plus B's new ones there.
__global__ void __launch_bounds__(256)
k_sum_tiles(int na, int nb, int tile_rows, const int32_t* __restrict__ a_rank, const int32_t* __restrict__ b_rank,
            const int64_t* __restrict__ u, const int32_t* __restrict__ a_row, const int32_t* __restrict__ a_col,
            const uint16_t* __restrict__ a_masks, const int32_t* __restrict__ a_rp, const int32_t* __restrict__ b_row,
            const int32_t* __restrict__ b_col, const uint16_t* __restrict__ b_masks, const int32_t* __restrict__ b_rp,
            int2* __restrict__ src, int32_t* __restrict__ s_row, int32_t* __restrict__ s_col,
            uint16_t* __restrict__ s_masks, int64_t* __restrict__ cnt, int64_t* __restrict__ s_rp)
{
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t n = (int64_t)na + nb;
    if (g <= tile_rows) s_rp[g] = (int64_t)a_rp[g] + u[b_rp[g]];
    if (g == n) cnt[na + u[nb]] = 0;
    if (g >= n) return;
    int64_t pos;
    int ia = -1, ib = -1;
    if (g < na) {
        ia = (int)g;
        const int rk = a_rank[ia];
        ib = rk >= 0 ? rk : -1;
        pos = ia + u[rk >= 0 ? rk : ~rk];
    } else {
        const int j = (int)(g - na);
        if (u[j + 1] == u[j]) return;               // A holds this key: its A tile's thread writes the union tile
        ib = j;
        pos = b_rank[j] + u[j];
    }
    uint4 m0 = make_uint4(0, 0, 0, 0), m1 = m0;
    if (ia >= 0) {
        const uint4* m4 = reinterpret_cast<const uint4*>(a_masks + (size_t)ia * 16);
        m0 = m4[0];
        m1 = m4[1];
    }
    if (ib >= 0) {
        const uint4* m4 = reinterpret_cast<const uint4*>(b_masks + (size_t)ib * 16);
        const uint4 x = m4[0], y = m4[1];
        m0 = make_uint4(m0.x | x.x, m0.y | x.y, m0.z | x.z, m0.w | x.w);
        m1 = make_uint4(m1.x | y.x, m1.y | y.y, m1.z | y.z, m1.w | y.w);
    }
    uint4* o4 = reinterpret_cast<uint4*>(s_masks + (size_t)pos * 16);
    o4[0] = m0;
    o4[1] = m1;
    src[pos] = make_int2(ia, ib);
    s_row[pos] = ia >= 0 ? a_row[ia] : b_row[ib];
    s_col[pos] = ia >= 0 ? a_col[ia] : b_col[ib];
    cnt[pos] = __popc(m0.x) + __popc(m0.y) + __popc(m0.z) + __popc(m0.w) + __popc(m1.x) + __popc(m1.y) + __popc(m1.z) +
               __popc(m1.w);
}

// The roundings of the contract, spelled out so that nvcc cannot contract alpha*a + beta*b into a fused multiply-add
__device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ double add_rn(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }

// Index of entry (r, c) in tile t of an operand, and whether the tile holds it
__device__ __forceinline__ bool operand_slot(int t, unsigned r, unsigned c, const uint32_t* __restrict__ nnz_ptr,
                                             const uint16_t* __restrict__ masks, const uint8_t* __restrict__ row_ptr,
                                             uint32_t* x)
{
    if (t < 0) return false;
    const unsigned m = masks[(size_t)t * 16 + r];
    *x = nnz_ptr[t] + row_ptr[(size_t)t * 16 + r] + __popc(m & ((1u << c) - 1u));
    return (m >> c) & 1u;
}

// S's values from A's and B's, one lane per value slot of S (pem_write_slots), into vals_t too when S's column-major
// view exists.  An entry of both operands is fl(fl(alpha*a) + fl(beta*b)), one of A only fl(alpha*a), one of B only
// fl(beta*b).
template <class T>
__global__ void __launch_bounds__(256)
k_add_vals(int cnt, const uint32_t* __restrict__ tile_nnz_ptr, const uint8_t* __restrict__ rc_idx,
           const int2* __restrict__ src, const uint32_t* __restrict__ col_rec, T alpha,
           const uint32_t* __restrict__ a_nnz_ptr, const uint16_t* __restrict__ a_masks,
           const uint8_t* __restrict__ a_row_ptr, const T* __restrict__ a_vals, T beta,
           const uint32_t* __restrict__ b_nnz_ptr, const uint16_t* __restrict__ b_masks,
           const uint8_t* __restrict__ b_row_ptr, const T* __restrict__ b_vals, T* __restrict__ vals,
           T* __restrict__ vals_t)
{
    pem_write_slots((int64_t)blockIdx.x * blockDim.x + threadIdx.x, threadIdx.x, cnt, tile_nnz_ptr, rc_idx, col_rec, vals,
                    vals_t, [=](uint32_t x, int64_t t) {
                        const unsigned rc = rc_idx[x];
                        const unsigned r = rc >> 4, c = rc & 15u;
                        const int2 st = src[t];
                        uint32_t xa = 0, xb = 0;
                        const bool in_a = operand_slot(st.x, r, c, a_nnz_ptr, a_masks, a_row_ptr, &xa);
                        const bool in_b = operand_slot(st.y, r, c, b_nnz_ptr, b_masks, b_row_ptr, &xb);
                        const T pa = in_a ? mul_rn(alpha, a_vals[xa]) : T(0);
                        const T pb = in_b ? mul_rn(beta, b_vals[xb]) : T(0);
                        return in_a && in_b ? add_rn(pa, pb) : in_a ? pa : pb;
                    });
}

}  // namespace

// The one kernel of pem_tiled_add_values, also the last step of pem_tiled_add
static int add_vals_launch(pem_ctx* ctx, pem_tiled* S, double alpha, const pem_tiled* A, double beta, const pem_tiled* B)
{
    if (!S->tiles) return PEM_OK;
    const int grid = pem_div_up(S->tiles, 256);        // a warp per 32 tiles
    pem_by_dtype(S->dtype, [&](auto v) {
        using VT = decltype(v);
        k_add_vals<VT><<<grid, 256, 0, ctx->stream>>>(
            S->tiles, S->tile_nnz_ptr, S->rc_idx, S->add_src, S->col_rec, (VT)alpha, A->tile_nnz_ptr, A->masks, A->row_ptr,
            pem_vals<VT>(A->vals), (VT)beta, B->tile_nnz_ptr, B->masks, B->row_ptr, pem_vals<VT>(B->vals),
            pem_vals<VT>(S->vals), pem_vals<VT>(S->vals_t));
    });
    PEM_LAUNCHED();
    return PEM_OK;
}

extern "C" {

int pem_tiled_add(pem_ctx* ctx, double alpha, const pem_tiled* A, double beta, const pem_tiled* B, pem_tiled** out)
{
    PEM_RANGE("pem_tiled_add");
    if (!ctx || !A || !B || !out) return PEM_ERR_ARG;
    *out = nullptr;
    if (A->rows != B->rows || A->cols != B->cols) return ctx->fail(PEM_ERR_ARG, "pem_tiled_add: the operands' shapes differ");
    if (A->dtype != B->dtype) return ctx->fail(PEM_ERR_ARG, "pem_tiled_add: the operands' value types differ");
    PEM_CK(cudaSetDevice(ctx->device));
    pem_tiled_ptr S = pem_tiled_new(ctx, A->dtype, A->rows, A->cols, 0);       // nnz: read back below
    S->origin = {PEM_BUILT_SUM, A->uid, B->uid};
    const int na = A->tiles, nb = B->tiles;
    const int64_t n = (int64_t)na + nb;
    int32_t *a_rank = nullptr, *b_rank = nullptr, *s_row = nullptr, *s_col = nullptr;
    int64_t *u = nullptr, *cnt = nullptr, *s_rp = nullptr;
    uint16_t* s_masks = nullptr;
    pem_guard g(ctx, a_rank, b_rank, u, s_row, s_col, s_masks, cnt, s_rp);

    // union tile list: ranks, the scan of B's new tiles, the union's size (read-back 1)
    int64_t ns = 0;
    if (n > 0) {
        PEM_TRY(pem_alloc(ctx, &a_rank, (size_t)na));
        PEM_TRY(pem_alloc(ctx, &b_rank, (size_t)nb));
        PEM_TRY(pem_alloc(ctx, &u, (size_t)nb + 1));
        k_sum_rank<<<pem_div_up(n + 1, 256), 256, 0, ctx->stream>>>(na, nb, A->tile_row_idx, A->tile_col_idx, A->tile_row_ptr,
                                                                   B->tile_row_idx, B->tile_col_idx, B->tile_row_ptr,
                                                                   a_rank, b_rank, u);
        PEM_LAUNCHED();
        PEM_TRY(pem_scan_exclusive_i64(ctx, u, (int64_t)nb + 1));
        PEM_CK(cudaMemcpyAsync(ctx->h_scalars, u + nb, 8, cudaMemcpyDeviceToHost, ctx->stream));
        PEM_CK(cudaStreamSynchronize(ctx->stream));
        ns = na + ctx->h_scalars[0];
    }
    if (ns >= (int64_t(1) << 31) - 1) return ctx->fail(PEM_ERR_LIMIT, "more than 2^31 tiles");
    S->tiles = (int32_t)ns;
    PEM_TRY(pem_alloc(ctx, &S->add_src, (size_t)ns));
    // the union as a result: tiles, masks, value offsets (read-back 2: nnz) and tile-row pointer
    if (n > 0) {
        PEM_TRY(pem_alloc(ctx, &s_row, (size_t)ns)); PEM_TRY(pem_alloc(ctx, &s_col, (size_t)ns));
        PEM_TRY(pem_alloc(ctx, &s_masks, (size_t)ns * 16));
        PEM_TRY(pem_alloc(ctx, &cnt, (size_t)ns + 1)); PEM_TRY(pem_alloc(ctx, &s_rp, (size_t)S->tile_rows + 1));
        k_sum_tiles<<<pem_div_up(std::max<int64_t>(n, S->tile_rows) + 1, 256), 256, 0, ctx->stream>>>(
            na, nb, S->tile_rows, a_rank, b_rank, u, A->tile_row_idx, A->tile_col_idx, A->masks, A->tile_row_ptr,
            B->tile_row_idx, B->tile_col_idx, B->masks, B->tile_row_ptr, S->add_src, s_row, s_col, s_masks, cnt, s_rp);
        PEM_LAUNCHED();
        PEM_TRY(pem_scan_exclusive_i64(ctx, cnt, ns + 1));
        PEM_CK(cudaMemcpyAsync(ctx->h_scalars, cnt + ns, 8, cudaMemcpyDeviceToHost, ctx->stream));
        PEM_CK(cudaStreamSynchronize(ctx->stream));
        S->nnz = ctx->h_scalars[0];
        pem_free(ctx, a_rank); pem_free(ctx, b_rank); pem_free(ctx, u);
    }
    if (S->nnz >= (int64_t(1) << 32) - 1) return ctx->fail(PEM_ERR_LIMIT, "nnz must be below 2^32-1 (32-bit tile value offsets)");
    pem_result U;
    U.dtype = S->dtype;
    U.rb = 0; U.re = S->tile_rows;
    U.rows = S->rows; U.cols = S->cols; U.tile_cols = S->tile_cols;
    U.tiles = ns; U.nnz = S->nnz;
    U.stage = 3;
    U.row_ptr = s_rp; U.tile_row = s_row; U.tile_col = s_col; U.masks = s_masks; U.tile_nnz_ptr = cnt;
    PEM_TRY(pem_operand_structure(ctx, &U, nullptr, S.get()));
    // the operands' values: a pending upload first
    PEM_TRY(pem_tiled_wait_vals(ctx, A));
    PEM_TRY(pem_tiled_wait_vals(ctx, B));
    PEM_TRY(add_vals_launch(ctx, S.get(), alpha, A, beta, B));
    PEM_TRY(pem_tiled_publish(ctx, S.get()));
    *out = S.release();
    return PEM_OK;
}

int pem_tiled_add_values(pem_ctx* ctx, pem_tiled* S, double alpha, const pem_tiled* A, double beta, const pem_tiled* B)
{
    PEM_RANGE("pem_tiled_add_values");
    if (!ctx || !S || !A || !B) return PEM_ERR_ARG;
    if (S->origin.kind != PEM_BUILT_SUM)
        return ctx->fail(PEM_ERR_ARG, "pem_tiled_add_values: the matrix was not built by pem_tiled_add");
    if (A->uid != S->origin.a_uid || B->uid != S->origin.b_uid)
        return ctx->fail(PEM_ERR_ARG, "pem_tiled_add_values: A and B are not the operands the sum was built from, in that order");
    PEM_CK(cudaSetDevice(ctx->device));
    PEM_TRY(pem_tiled_wait_vals(ctx, A));
    PEM_TRY(pem_tiled_wait_vals(ctx, B));
    return add_vals_launch(ctx, S, alpha, A, beta, B);
}

}  // extern "C"
