// Results as operands: a complete C (or panel of C) -> an independent tiled matrix, without the COO round trip.
//
// C is already tiled: its C' tiles are ordered by (tile row, tile column), its masks are the row masks a pem_tiled
// holds, and its values are tile-major and row-major inside a tile, the layout of pem_tiled::vals.  So the handle
// pem_convert_coo would build from pem_result_to_coo(C) comes out of one thread per tile (masks, column masks, row
// pointers, occupancy words, tile indices and offsets) and one pass over C's rows (the (r, c) byte of every value and
// its position in C's row-major order, the value map): no sort.  Empty C' tiles (PEM_OPT_KEEP_EMPTY_TILES) are
// dropped; they hold no values, so every value keeps its slot and the values are one copy.
#include <cub/device/device_select.cuh>
#include <thrust/iterator/counting_iterator.h>

#include "engine.cuh"

namespace {

// predicate of the keep-empty compaction: C' tile t holds a nonzero
struct TileHasEntries {
    const uint4* masks;
    __device__ __forceinline__ bool operator()(int32_t t) const
    {
        const uint4 a = masks[2 * (size_t)t], b = masks[2 * (size_t)t + 1];
        return (a.x | a.y | a.z | a.w | b.x | b.y | b.z | b.w) != 0u;
    }
};

// One thread per kept tile i (C' tile keep[i], or i when nothing was dropped); threads up to tile_rows also write the
// tile-row pointers outside the panel [rb, re), which hold no tile.  Thread cnt writes the end of the value offsets.
__global__ void __launch_bounds__(128)
k_operand_tiles(int cnt, const int32_t* __restrict__ keep, const uint16_t* __restrict__ c_masks,
                const int32_t* __restrict__ c_tile_row, const int32_t* __restrict__ c_tile_col,
                const int64_t* __restrict__ c_nnz_ptr, uint32_t nnz, int rb, int re, int tile_rows,
                uint32_t* __restrict__ nnz_ptr, uint16_t* __restrict__ masks, uint16_t* __restrict__ masks_t,
                uint8_t* __restrict__ row_ptr, int32_t* __restrict__ tile_row, int32_t* __restrict__ tile_col,
                int32_t* __restrict__ tile_row_ptr, uint16_t* __restrict__ col_occ, uint16_t* __restrict__ row_occ)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i <= tile_rows && (i < rb || i > re || cnt == 0)) tile_row_ptr[i] = i < rb ? 0 : cnt;
    if (i == cnt) nnz_ptr[cnt] = nnz;
    if (i >= cnt) return;
    const int s = keep ? keep[i] : i;
    const uint4* m4 = reinterpret_cast<const uint4*>(c_masks + (size_t)s * 16);
    const uint4 a = m4[0], b = m4[1];
    reinterpret_cast<uint4*>(masks + (size_t)i * 16)[0] = a;
    reinterpret_cast<uint4*>(masks + (size_t)i * 16)[1] = b;
    const unsigned w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    unsigned m[16], packed[4] = {0, 0, 0, 0};
    unsigned run = 0, cols = 0, rows = 0;
#pragma unroll
    for (int r = 0; r < 16; ++r) {
        m[r] = (w[r >> 1] >> ((r & 1) * 16)) & 0xFFFFu;
        packed[r >> 2] |= run << (8 * (r & 3));
        run += __popc(m[r]);
        cols |= m[r];
        rows |= m[r] ? 1u << r : 0u;
    }
    *reinterpret_cast<uint4*>(row_ptr + (size_t)i * 16) = make_uint4(packed[0], packed[1], packed[2], packed[3]);
    col_occ[i] = (uint16_t)cols;
    row_occ[i] = (uint16_t)rows;
    // 16x16 bit transpose in registers: swap the off-diagonal j x j blocks of every 2j x 2j block, j = 8, 4, 2, 1
#pragma unroll
    for (int l = 0; l < 4; ++l) {
        const int j = 8 >> l;
        const unsigned lo = l == 0 ? 0x00FFu : l == 1 ? 0x0F0Fu : l == 2 ? 0x3333u : 0x5555u;
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            if (k & j) continue;
            const unsigned t = ((m[k] >> j) ^ m[k | j]) & lo;
            m[k] ^= t << j;
            m[k | j] ^= t;
        }
    }
    uint4* t4 = reinterpret_cast<uint4*>(masks_t + (size_t)i * 16);
    t4[0] = make_uint4(m[0] | m[1] << 16, m[2] | m[3] << 16, m[4] | m[5] << 16, m[6] | m[7] << 16);
    t4[1] = make_uint4(m[8] | m[9] << 16, m[10] | m[11] << 16, m[12] | m[13] << 16, m[14] | m[15] << 16);
    const int tr = c_tile_row[s];
    tile_row[i] = tr;
    tile_col[i] = c_tile_col[s];
    nnz_ptr[i] = (uint32_t)c_nnz_ptr[s];
    // tile-level CSR row pointer: this tile opens every tile row after the previous kept tile's, from the panel's first
    const int prev = i ? c_tile_row[keep ? keep[i - 1] : i - 1] : rb - 1;
    for (int r = prev + 1; r <= tr; ++r) tile_row_ptr[r] = i;
    if (i == cnt - 1)
        for (int r = tr + 1; r <= re; ++r) tile_row_ptr[r] = cnt;
}

// 16 lanes per tile row of C, lane r = matrix row: walks the row's entries in column order (the tiles of a tile row
// are ordered by tile column), as k_export_fill does, and writes for each value slot its (r, c) byte and its position
// in C's row-major order (pos starts at the row's pointer)
__global__ void __launch_bounds__(256)
k_operand_slots(int n_tile_rows, const int64_t* __restrict__ c_row_ptr, const uint16_t* __restrict__ c_masks,
                const int64_t* __restrict__ c_nnz_ptr, const int64_t* __restrict__ row_pos,
                uint8_t* __restrict__ rc_idx, uint32_t* __restrict__ val_pos)
{
    const int g = (blockIdx.x * blockDim.x + threadIdx.x) >> 4;
    const int r = threadIdx.x & 15;
    if (g >= n_tile_rows) return;
    const unsigned grp = 0xFFFFu << (threadIdx.x & 16);  // the 16 lanes of this group inside the warp
    uint32_t pos = (uint32_t)row_pos[(int64_t)g * 16 + r];
    for (int64_t t = c_row_ptr[g]; t < c_row_ptr[g + 1]; ++t) {
        unsigned m = c_masks[t * 16 + r];
        // first slot of row r inside the tile = popcounts of rows < r
        const int pc = __popc(m);
        int incl = pc;
#pragma unroll
        for (int o = 1; o < 16; o <<= 1) {
            const int v = __shfl_up_sync(grp, incl, o, 16);
            if (r >= o) incl += v;
        }
        uint32_t x = (uint32_t)c_nnz_ptr[t] + (uint32_t)(incl - pc);
        while (m) {
            const int c = __ffs(m) - 1;
            m &= m - 1;
            rc_idx[x] = (uint8_t)((r << 4) | c);
            val_pos[x] = pos;
            ++x;
            ++pos;
        }
    }
}

}  // namespace

// The structure of T from a result-shaped tile list C (tile-row pointer over [rb, re), tile rows and columns, row masks,
// value offsets): the arrays of T, T->vals included, allocated for T->tiles tiles (C' tile keep[i] for tile i, or tile i
// when keep is null) and T->nnz values, and every array but vals written.  T's shape is set by the caller.  Stream order;
// the caller fills vals and publishes T.  pem_result_to_tiled and pem_tiled_add (sum.cu).
int pem_operand_structure(pem_ctx* ctx, const pem_result* C, const int32_t* keep, pem_tiled* T)
{
    const int ntr = C->re - C->rb;
    const int64_t cnt = T->tiles;
    int64_t* row_pos = nullptr;
    pem_guard g(ctx, row_pos);
    PEM_TRY(pem_tiled_alloc(ctx, T));

    const int64_t threads = std::max<int64_t>(cnt, T->tile_rows) + 1;
    k_operand_tiles<<<pem_div_up(threads, 128), 128, 0, ctx->stream>>>(
        (int)cnt, keep, C->masks, C->tile_row, C->tile_col, C->tile_nnz_ptr, (uint32_t)C->nnz, C->rb, C->re, T->tile_rows,
        T->tile_nnz_ptr, T->masks, T->masks_t, T->row_ptr, T->tile_row_idx, T->tile_col_idx, T->tile_row_ptr, T->col_occ,
        T->row_occ);
    PEM_LAUNCHED();
    if (T->nnz) {
        // first position of every row of the panel in C's row-major order: the export's row count and scan
        PEM_TRY(pem_alloc(ctx, &row_pos, (size_t)ntr * 16 + 1));
        PEM_TRY(pem_result_to_coo_device(ctx, C, nullptr, nullptr, nullptr, row_pos));
        k_operand_slots<<<pem_div_up((int64_t)ntr * 16, 256), 256, 0, ctx->stream>>>(
            ntr, C->row_ptr, C->masks, C->tile_nnz_ptr, row_pos, T->rc_idx, T->val_pos);
        PEM_LAUNCHED();
    }
    return PEM_OK;
}

extern "C" {

int pem_result_to_tiled(pem_ctx* ctx, const pem_result* C, pem_tiled** out)
{
    PEM_RANGE("pem_result_to_tiled");
    if (!ctx || !C || !out) return PEM_ERR_ARG;
    *out = nullptr;
    if (C->stage != 3) return ctx->fail(PEM_ERR_ARG, "pem_result_to_tiled needs a complete result (step 3 done)");
    if (C->nnz >= (int64_t(1) << 32) - 1) return ctx->fail(PEM_ERR_LIMIT, "nnz must be below 2^32-1 (32-bit tile value offsets)");
    if (C->tiles >= (int64_t(1) << 31) - 1) return ctx->fail(PEM_ERR_LIMIT, "more than 2^31 tiles");
    PEM_CK(cudaSetDevice(ctx->device));
    pem_tiled_ptr T = pem_tiled_new(ctx, C->dtype, C->rows, C->cols, C->nnz);
    T->origin = {PEM_BUILT_RESULT, C->a_uid, C->b_uid, C->rb, C->re};
    int32_t* keep = nullptr;                  // kept C' tile of every tile of T (keep-empty results only)
    char* tmp = nullptr;
    pem_guard g(ctx, keep, tmp);

    // a result of the default mode holds non-empty tiles only; otherwise the empty ones are dropped here (one read-back)
    int64_t cnt = C->tiles;
    if (C->keep_empty && C->tiles > 0) {
        thrust::counting_iterator<int32_t> iota(0);
        TileHasEntries pred{reinterpret_cast<const uint4*>(C->masks)};
        int64_t* d_count = ctx->d_scalars + SC_COUNT;
        size_t tb = 0;
        PEM_CK(cub::DeviceSelect::If(nullptr, tb, iota, keep, d_count, C->tiles, pred, ctx->stream));
        PEM_TRY(pem_alloc(ctx, &keep, (size_t)C->tiles));
        PEM_TRY(pem_alloc(ctx, &tmp, tb));
        PEM_CK(cub::DeviceSelect::If(tmp, tb, iota, keep, d_count, C->tiles, pred, ctx->stream));
        ctx->launches += 2;
        PEM_CK(cudaMemcpyAsync(ctx->h_scalars, d_count, 8, cudaMemcpyDeviceToHost, ctx->stream));
        PEM_CK(cudaStreamSynchronize(ctx->stream));
        cnt = ctx->h_scalars[0];
        pem_free(ctx, tmp);
    }
    T->tiles = (int32_t)cnt;
    PEM_TRY(pem_operand_structure(ctx, C, keep, T.get()));
    // every value keeps its slot: empty tiles hold none
    if (T->nnz) PEM_CK(cudaMemcpyAsync(T->vals, C->vals, (size_t)T->nnz * pem_vsize(T->dtype), cudaMemcpyDeviceToDevice, ctx->stream));
    PEM_TRY(pem_tiled_publish(ctx, T.get()));
    *out = T.release();
    return PEM_OK;
}

int pem_tiled_refresh_from_result(pem_ctx* ctx, pem_tiled* T, const pem_result* C)
{
    PEM_RANGE("pem_tiled_refresh_from_result");
    if (!ctx || !T || !C) return PEM_ERR_ARG;
    const pem_origin& o = T->origin;
    if (o.kind != PEM_BUILT_RESULT)
        return ctx->fail(PEM_ERR_ARG, "pem_tiled_refresh_from_result: the matrix was not built by pem_result_to_tiled "
                                      "(refresh it with pem_tiled_set_values)");
    if (C->stage != 3) return ctx->fail(PEM_ERR_ARG, "pem_tiled_refresh_from_result needs a complete result (step 3 done)");
    if (C->a_uid != o.a_uid || C->b_uid != o.b_uid || C->rb != o.rb || C->re != o.re)
        return ctx->fail(PEM_ERR_ARG, "pem_tiled_refresh_from_result: the result is not of the product the matrix was built from");
    PEM_CK(cudaSetDevice(ctx->device));
    return pem_tiled_write_slots(ctx, T, C->vals);
}

}  // extern "C"
