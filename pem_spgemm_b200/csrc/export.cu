// Tiled C -> COO/CSR sorted by (row, col), and a device-side checksum.
//
// Replaces /root/reference/spgemm.cu:1493-1543: sanitize_C (:663-695) followed by a
// thrust::stable_sort of (row, col, val) tuples over all of C.  The tiles of a tile row are
// already ordered by tile column and the entries of a tile are row-major, so no sort is needed:
// 16 lanes (one per row of the tile row) walk the tile row's tiles in order; lane r counts, then
// places, the entries of matrix row 16*i + r.  The row pointer comes out as a by-product (CSR).
#include <algorithm>
#include <vector>

#include "engine.cuh"

namespace {

// 16 lanes per tile row; lane r sums popc(Cmask[t][r]) over the row's tiles.
__global__ void __launch_bounds__(256)
k_export_count(int n_tile_rows, const int64_t* __restrict__ c_row_ptr, const uint16_t* __restrict__ Cmasks,
               int64_t* __restrict__ row_cnt)
{
    int g = (blockIdx.x * blockDim.x + threadIdx.x) >> 4;
    int r = threadIdx.x & 15;
    if (g >= n_tile_rows) return;
    int64_t cnt = 0;
    for (int64_t t = c_row_ptr[g]; t < c_row_ptr[g + 1]; ++t) cnt += __popc((unsigned)Cmasks[t * 16 + r]);
    row_cnt[(int64_t)g * 16 + r] = cnt;
}

template <class T>
__global__ void __launch_bounds__(256)
k_export_fill(int n_tile_rows, int rb, const int64_t* __restrict__ c_row_ptr, const int32_t* __restrict__ c_tile_col,
              const uint16_t* __restrict__ Cmasks, const int64_t* __restrict__ c_tile_nnz_ptr,
              const T* __restrict__ C_vals, const int64_t* __restrict__ row_ptr,
              int32_t* __restrict__ rows, int32_t* __restrict__ cols, T* __restrict__ vals)
{
    int g = (blockIdx.x * blockDim.x + threadIdx.x) >> 4;
    int r = threadIdx.x & 15;
    if (g >= n_tile_rows) return;
    const unsigned grp = 0xFFFFu << (threadIdx.x & 16);  // the 16 lanes of this group inside the warp
    int64_t pos = row_ptr[(int64_t)g * 16 + r];
    const int row = (rb + g) * 16 + r;
    for (int64_t t = c_row_ptr[g]; t < c_row_ptr[g + 1]; ++t) {
        unsigned m = Cmasks[t * 16 + r];
        // offset of row r inside the tile = popcounts of rows < r (segmented inclusive scan - own)
        int pc = __popc(m), incl = pc;
#pragma unroll
        for (int o = 1; o < 16; o <<= 1) {
            int v = __shfl_up_sync(grp, incl, o, 16);
            if (r >= o) incl += v;
        }
        int64_t src = c_tile_nnz_ptr[t] + (incl - pc);
        const int cbase = c_tile_col[t] * 16;
        while (m) {
            int c = __ffs(m) - 1;
            m &= m - 1;
            if (rows) rows[pos] = row;
            if (cols) cols[pos] = cbase + c;
            if (vals) vals[pos] = C_vals[src];
            ++src;
            ++pos;
        }
    }
}

// deterministic two-level reduction of sum and sum|.|
template <class T>
__global__ void __launch_bounds__(256)
k_checksum_partial(const T* __restrict__ v, int64_t n, double* __restrict__ part)
{
    __shared__ double s1[8], s2[8];
    double a = 0, b = 0;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
        double x = (double)v[i];
        a += x;
        b += fabs(x);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b += __shfl_xor_sync(0xffffffffu, b, o);
    }
    if ((threadIdx.x & 31) == 0) { s1[threadIdx.x >> 5] = a; s2[threadIdx.x >> 5] = b; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double x = 0, y = 0;
        for (int w = 0; w < 8; ++w) { x += s1[w]; y += s2[w]; }
        part[2 * blockIdx.x] = x;
        part[2 * blockIdx.x + 1] = y;
    }
}

}  // namespace

extern "C" {

int pem_result_to_coo_device(pem_ctx* ctx, const pem_result* C, int32_t* d_rows, int32_t* d_cols,
                             double* d_vals, int64_t* d_row_ptr)
{
    if (!ctx || !C) return PEM_ERR_ARG;
    if (C->stage < 2 || (d_vals && C->stage < 3)) return ctx->fail(PEM_ERR_ARG, "result is not complete");
    PEM_CK(cudaSetDevice(ctx->device));
    const int ntr = C->re - C->rb;
    const size_t nrow = (size_t)ntr * 16;
    int64_t* own_rp = nullptr;                 // the row pointer is a temporary unless the caller wants it
    pem_guard g(ctx, own_rp);
    if (!d_row_ptr) PEM_TRY(pem_alloc(ctx, &own_rp, nrow + 1));
    int64_t* rp = d_row_ptr ? d_row_ptr : own_rp;
    PEM_CK(cudaMemsetAsync(rp, 0, (nrow + 1) * 8, ctx->stream));
    if (ntr > 0 && C->tiles > 0) {
        k_export_count<<<pem_div_up((int64_t)ntr * 16, 256), 256, 0, ctx->stream>>>(ntr, C->row_ptr, C->masks, rp);
        PEM_LAUNCHED();
    }
    PEM_TRY(pem_scan_exclusive_i64(ctx, rp, (int64_t)nrow + 1));
    if (ntr > 0 && C->tiles > 0 && (d_rows || d_cols || d_vals)) {
        if (C->dtype == PEM_F32)      // d_vals then points at floats
            k_export_fill<float><<<pem_div_up((int64_t)ntr * 16, 256), 256, 0, ctx->stream>>>(
                ntr, C->rb, C->row_ptr, C->tile_col, C->masks, C->tile_nnz_ptr, reinterpret_cast<const float*>(C->vals), rp,
                d_rows, d_cols, reinterpret_cast<float*>(d_vals));
        else
            k_export_fill<double><<<pem_div_up((int64_t)ntr * 16, 256), 256, 0, ctx->stream>>>(
                ntr, C->rb, C->row_ptr, C->tile_col, C->masks, C->tile_nnz_ptr, C->vals, rp, d_rows, d_cols, d_vals);
        PEM_LAUNCHED();
    }
    pem_free(ctx, own_rp);
    return PEM_OK;
}

static int result_to_coo_any(pem_ctx* ctx, const pem_result* C, int32_t* rows, int32_t* cols, void* vals, int dtype)
{
    PEM_RANGE("pem_result_to_coo");
    if (!ctx || !C) return PEM_ERR_ARG;
    if (vals && C->dtype != dtype)
        return ctx->fail(PEM_ERR_ARG, C->dtype == PEM_F32 ? "fp32 result: use pem_result_to_coo_f32" : "fp64 result: use pem_result_to_coo");
    const size_t vsz = pem_vsize(C->dtype);
    int32_t *dr = nullptr, *dc = nullptr;
    double* dv = nullptr;
    pem_guard g(ctx, dr, dc, dv);
    size_t n = (size_t)C->nnz;
    if (rows) PEM_TRY(pem_alloc(ctx, &dr, n));
    if (cols) PEM_TRY(pem_alloc(ctx, &dc, n));
    if (vals) PEM_TRY(pem_alloc_bytes(ctx, (void**)&dv, std::max<size_t>(1, n * vsz)));
    PEM_TRY(pem_result_to_coo_device(ctx, C, dr, dc, dv, nullptr));
    if (n) {
        if (rows) PEM_CK(cudaMemcpyAsync(rows, dr, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
        if (cols) PEM_CK(cudaMemcpyAsync(cols, dc, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
        if (vals) PEM_CK(cudaMemcpyAsync(vals, dv, n * vsz, cudaMemcpyDeviceToHost, ctx->stream));
        PEM_CK(cudaStreamSynchronize(ctx->stream));
    }
    return PEM_OK;
}

int pem_result_to_coo(pem_ctx* ctx, const pem_result* C, int32_t* rows, int32_t* cols, double* vals)
{
    return result_to_coo_any(ctx, C, rows, cols, vals, PEM_F64);
}

int pem_result_to_coo_f32(pem_ctx* ctx, const pem_result* C, int32_t* rows, int32_t* cols, float* vals)
{
    return result_to_coo_any(ctx, C, rows, cols, vals, PEM_F32);
}

int pem_result_to_csr(pem_ctx* ctx, const pem_result* C, int64_t* row_ptr, int32_t* cols, double* vals)
{
    PEM_RANGE("pem_result_to_csr");
    if (!ctx || !C) return PEM_ERR_ARG;
    if (vals && C->dtype != PEM_F64) return ctx->fail(PEM_ERR_ARG, "pem_result_to_csr returns fp64 values: use pem_result_to_coo_f32 for an fp32 result");
    const int64_t first_row = (int64_t)C->rb * 16;
    const int64_t nrows = std::max<int64_t>(0, std::min<int64_t>(C->rows, (int64_t)C->re * 16) - first_row);
    int32_t* dc = nullptr;
    double* dv = nullptr;
    int64_t* drp = nullptr;
    pem_guard g(ctx, dc, dv, drp);
    const size_t n = (size_t)C->nnz;
    if (cols) PEM_TRY(pem_alloc(ctx, &dc, n));
    if (vals) PEM_TRY(pem_alloc(ctx, &dv, n));
    PEM_TRY(pem_alloc(ctx, &drp, (size_t)(C->re - C->rb) * 16 + 1));
    PEM_TRY(pem_result_to_coo_device(ctx, C, nullptr, dc, dv, drp));
    // rows past the matrix edge (last tile row) are empty: their pointers equal nnz, so the first nrows + 1 entries are the CSR pointer
    if (row_ptr) PEM_CK(cudaMemcpyAsync(row_ptr, drp, ((size_t)nrows + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
    if (cols && n) PEM_CK(cudaMemcpyAsync(cols, dc, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (vals && n) PEM_CK(cudaMemcpyAsync(vals, dv, n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    PEM_CK(cudaStreamSynchronize(ctx->stream));
    return PEM_OK;
}

int pem_result_checksum(pem_ctx* ctx, const pem_result* C, double* sum, double* abs_sum)
{
    if (!ctx || !C) return PEM_ERR_ARG;
    if (C->stage < 3) return ctx->fail(PEM_ERR_ARG, "result has no values yet");
    PEM_CK(cudaSetDevice(ctx->device));
    const int nb = 1024;
    double* part = nullptr;
    pem_guard g(ctx, part);
    PEM_TRY(pem_alloc(ctx, &part, (size_t)2 * nb));
    if (C->dtype == PEM_F32) k_checksum_partial<float><<<nb, 256, 0, ctx->stream>>>(reinterpret_cast<const float*>(C->vals), C->nnz, part);
    else k_checksum_partial<double><<<nb, 256, 0, ctx->stream>>>(C->vals, C->nnz, part);
    PEM_LAUNCHED();
    std::vector<double> h((size_t)2 * nb);
    PEM_CK(cudaMemcpyAsync(h.data(), part, h.size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
    PEM_CK(cudaStreamSynchronize(ctx->stream));
    pem_free(ctx, part);
    double a = 0, b = 0;
    for (int i = 0; i < nb; ++i) { a += h[2 * (size_t)i]; b += h[2 * (size_t)i + 1]; }
    if (sum) *sum = a;
    if (abs_sum) *abs_sum = b;
    return PEM_OK;
}

}  // extern "C"
