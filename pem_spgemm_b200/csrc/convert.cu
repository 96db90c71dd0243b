// COO -> 16x16 tiled CSR on the GPU, plus flop counting and the flop-balanced panel split.
//
// Replaces /root/reference/spgemm.cu:821-1066: decide_which_tile (:112-135), the thrust
// sort / unique_count / reduce_by_key / scan / unique census (:866-892), the tuple merge sort
// to CSR (:894-928), generate_tiles_csr with its 256 binary searches per tile (:137-226),
// __transpose_B_mask (:228-258) and the tile-level CSR build (:985-1031).
//
// B200 design: ONE radix sort.  Every nonzero gets a 64-bit key
//     (tileRow, tileCol, r, c)  packed as  tileRow << (cb+8) | tileCol << 8 | r << 4 | c
// and is sorted together with its value over exactly the bits in use (8 + cb + rb, 5-6 radix
// passes).  The sorted value array IS the tiled value array (tile-major, row-major inside a
// tile); tile boundaries are the positions where key>>8 changes; one thread per tile then folds
// its keys' low bytes into the row masks, column masks, row pointers and occupancy words with
// 64-bit register bit-sets (no binary search, no shared memory, no CSR intermediate).
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_select.cuh>
#include <cub/iterator/counting_input_iterator.cuh>

#include <chrono>
#include <vector>

#include "engine.cuh"

namespace {

inline int h_bits_for(int64_t n)
{
    int b = 1;
    while ((int64_t(1) << b) < n) ++b;
    return b;
}

// One thread per nonzero: range check, optional transpose, key packing.
__global__ void __launch_bounds__(256)
k_make_keys(const int32_t* __restrict__ I, const int32_t* __restrict__ J, int64_t nnz,
            int rows, int cols, int transpose, int cb, uint64_t* __restrict__ keys,
            uint32_t* __restrict__ pos, int64_t* __restrict__ scalars)
{
    int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; e < nnz; e += stride) {
        int i = I[e], j = J[e];
        if (transpose) { int t = i; i = j; j = t; }
        uint64_t key;
        if ((unsigned)i >= (unsigned)rows || (unsigned)j >= (unsigned)cols) {
            atomicOr((unsigned long long*)&scalars[SC_ERR], 1ull);
            key = 0;
        } else {
            key = ((uint64_t)(i >> 4) << (cb + 8)) | ((uint64_t)(j >> 4) << 8) | (uint64_t)(((i & 15) << 4) | (j & 15));
        }
        keys[e] = key;
        pos[e] = (uint32_t)e;
    }
}

// (r<<4)|c of every value = low byte of its sorted key; the value itself is fetched through the
// sorted original position (the sort carries 4-byte positions, not 8-byte values, and the values'
// host->device copy overlaps it)
__global__ void __launch_bounds__(256)
k_rc_idx(const uint64_t* __restrict__ keys, int64_t nnz, uint8_t* __restrict__ rc)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e < nnz) rc[e] = (uint8_t)(keys[e] & 255u);
}
template <class T>
__global__ void __launch_bounds__(256)
k_gather_vals(const uint32_t* __restrict__ pos, const T* __restrict__ V, int64_t nnz, T* __restrict__ vals)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e < nnz) vals[e] = V[pos[e]];
}

// CSR input: row index of nonzero e = last row whose pointer is <= e (binary search; rows of any length)
__global__ void __launch_bounds__(256)
k_csr_rows(const int32_t* __restrict__ rp, int rows, int64_t nnz, int32_t* __restrict__ I)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= nnz) return;
    int lo = 0, hi = rows;                      // invariant: rp[lo] <= e < rp[hi]
    while (hi - lo > 1) {
        const int mid = (int)(((int64_t)lo + hi) >> 1);
        if ((int64_t)rp[mid] <= e) lo = mid; else hi = mid;
    }
    I[e] = lo;
}

// predicate for the tile census: position e starts a new tile
struct HeadPred {
    const uint64_t* keys;
    __device__ __forceinline__ bool operator()(uint32_t e) const
    {
        return e == 0 || (keys[e] >> 8) != (keys[e - 1] >> 8);
    }
};

__device__ __forceinline__ void set_bit256(uint64_t (&w)[4], unsigned b)
{
    uint64_t bit = 1ull << (b & 63);
    unsigned wi = b >> 6;
    w[0] |= wi == 0 ? bit : 0ull;
    w[1] |= wi == 1 ? bit : 0ull;
    w[2] |= wi == 2 ? bit : 0ull;
    w[3] |= wi == 3 ? bit : 0ull;
}

__device__ __forceinline__ unsigned fold16(const uint64_t (&w)[4])
{
    uint64_t x = w[0] | w[1] | w[2] | w[3];
    x |= x >> 32;
    x |= x >> 16;
    return (unsigned)(x & 0xFFFFu);
}

// One thread per tile.  keys are sorted; start[t] is the first nonzero of tile t.
__global__ void __launch_bounds__(128)
k_build_tiles(const uint64_t* __restrict__ keys, uint32_t* __restrict__ start, int cnt, uint32_t nnz,
              int cb, int tile_rows,
              uint16_t* __restrict__ masks, uint16_t* __restrict__ masks_t, uint8_t* __restrict__ row_ptr,
              int32_t* __restrict__ tile_col, int32_t* __restrict__ tile_row, int32_t* __restrict__ tile_row_ptr,
              uint16_t* __restrict__ col_occ, uint16_t* __restrict__ row_occ, int64_t* __restrict__ scalars)
{
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= cnt) return;
    uint32_t s = start[t];
    uint32_t e = (t + 1 < cnt) ? start[t + 1] : nnz;
    uint64_t w[4] = {0, 0, 0, 0}, wt[4] = {0, 0, 0, 0};
    uint64_t k0 = keys[s], prev = ~0ull;
    bool dup = false;
    for (uint32_t x = s; x < e; ++x) {
        uint64_t k = keys[x];
        dup |= (k == prev);
        prev = k;
        unsigned rc = (unsigned)(k & 255u);
        set_bit256(w, rc);                                  // bit r*16+c : row masks
        set_bit256(wt, ((rc & 15u) << 4) | (rc >> 4));      // bit c*16+r : column masks
    }
    if (dup) atomicOr((unsigned long long*)&scalars[SC_ERR], 2ull);

    // uint16 mask[16] in memory == four little-endian 64-bit words
    uint4* m4 = reinterpret_cast<uint4*>(masks + (size_t)t * 16);
    m4[0] = make_uint4((unsigned)w[0], (unsigned)(w[0] >> 32), (unsigned)w[1], (unsigned)(w[1] >> 32));
    m4[1] = make_uint4((unsigned)w[2], (unsigned)(w[2] >> 32), (unsigned)w[3], (unsigned)(w[3] >> 32));
    uint4* t4 = reinterpret_cast<uint4*>(masks_t + (size_t)t * 16);
    t4[0] = make_uint4((unsigned)wt[0], (unsigned)(wt[0] >> 32), (unsigned)wt[1], (unsigned)(wt[1] >> 32));
    t4[1] = make_uint4((unsigned)wt[2], (unsigned)(wt[2] >> 32), (unsigned)wt[3], (unsigned)(wt[3] >> 32));

    // row pointers: exclusive scan of the 16 row popcounts, one byte each (max 240)
    unsigned rp[4];
    unsigned run = 0;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        unsigned word = 0;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            int r = q * 4 + b;
            word |= run << (8 * b);
            run += __popcll(w[r >> 2] & (0xFFFFull << ((r & 3) * 16)));
        }
        rp[q] = word;
    }
    *reinterpret_cast<uint4*>(row_ptr + (size_t)t * 16) = make_uint4(rp[0], rp[1], rp[2], rp[3]);

    col_occ[t] = (uint16_t)fold16(w);
    row_occ[t] = (uint16_t)fold16(wt);

    int tr = (int)(k0 >> (cb + 8));
    int tc = (int)((k0 >> 8) & ((1ull << cb) - 1));
    tile_col[t] = tc;
    tile_row[t] = tr;
    // tile-level CSR row pointer: this tile opens every tile row after the previous tile's
    int prev_tr = (t == 0) ? -1 : (int)(keys[start[t - 1]] >> (cb + 8));
    for (int r = prev_tr + 1; r <= tr; ++r) tile_row_ptr[r] = t;
    if (t == cnt - 1) {
        for (int r = tr + 1; r <= tile_rows; ++r) tile_row_ptr[r] = cnt;
        start[cnt] = nnz;
    }
}

// per-row nonzero counts of a tiled matrix (thread per tile, 16 atomics at most)
__global__ void __launch_bounds__(256)
k_row_nnz(const uint16_t* __restrict__ masks, const int32_t* __restrict__ tile_row, int cnt,
          uint32_t* __restrict__ row_nnz)
{
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= cnt) return;
    const uint4* m4 = reinterpret_cast<const uint4*>(masks + (size_t)t * 16);
    uint4 a = m4[0], b = m4[1];
    unsigned w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    int base = tile_row[t] * 16;
#pragma unroll
    for (int r = 0; r < 16; ++r) {
        unsigned m = (w[r >> 1] >> ((r & 1) * 16)) & 0xFFFFu;
        if (m) atomicAdd(&row_nnz[base + r], (unsigned)__popc(m));
    }
}

// flop of one A tile = sum_k (nnz of A column k in the tile) * nnz(B row 16*tc + k); summed per tile row
__global__ void __launch_bounds__(256)
k_tile_flop(const uint16_t* __restrict__ masks_t, const int32_t* __restrict__ tile_row,
            const int32_t* __restrict__ tile_col, int cnt, const uint32_t* __restrict__ b_row_nnz, int b_rows,
            unsigned long long* __restrict__ tile_row_flop)
{
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= cnt) return;
    const uint4* m4 = reinterpret_cast<const uint4*>(masks_t + (size_t)t * 16);
    uint4 a = m4[0], b = m4[1];
    unsigned w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    int base = tile_col[t] * 16;
    unsigned long long f = 0;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        unsigned m = (w[k >> 1] >> ((k & 1) * 16)) & 0xFFFFu;
        if (m && base + k < b_rows) f += (unsigned long long)__popc(m) * b_row_nnz[base + k];
    }
    if (f) atomicAdd(&tile_row_flop[tile_row[t]], f);
}

// ---- row slices (see pem_tiled::srow_ptr) ------------------------------------------------------
// count: thread per tile, one atomic per occupied row of the tile
__global__ void __launch_bounds__(256)
k_srow_count(const uint16_t* __restrict__ row_occ, const int32_t* __restrict__ tile_row, int cnt,
             unsigned long long* __restrict__ srow_cnt)
{
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= cnt) return;
    unsigned occ = row_occ[t];
    const size_t base = (size_t)tile_row[t] * 16;
    while (occ) {
        const int r = __ffs(occ) - 1;
        occ &= occ - 1;
        atomicAdd(&srow_cnt[base + r], 1ull);
    }
}

// fill: thread per tile; every occupied row of the tile claims the next slot of its slice.  The order
// of the tiles inside a slice is irrelevant: step 1 sorts the expanded pairs by (C' row, tile column)
// and two tiles of one slice never share a tile column, so the result does not depend on it.
__global__ void __launch_bounds__(256)
k_srow_fill(const uint16_t* __restrict__ row_occ, const int32_t* __restrict__ tile_row, int cnt,
            const int64_t* __restrict__ srow_ptr, unsigned* __restrict__ cursor, int32_t* __restrict__ srow_tile)
{
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= cnt) return;
    unsigned occ = row_occ[t];
    const size_t base = (size_t)tile_row[t] * 16;
    while (occ) {
        const int r = __ffs(occ) - 1;
        occ &= occ - 1;
        srow_tile[srow_ptr[base + r] + atomicAdd(&cursor[base + r], 1u)] = t;
    }
}

// ---- step-3 views (see pem_tiled::row_rec) -----------------------------------------------------
__global__ void __launch_bounds__(256)
k_row_rec(const uint16_t* __restrict__ masks, const uint8_t* __restrict__ row_ptr, int64_t n, uint32_t* __restrict__ rec)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) rec[i] = (uint32_t)masks[i] | ((uint32_t)row_ptr[i] << 16);
}

// thread per tile: column pointers from the column masks, then every value goes to its column-major slot
template <class T>
__global__ void __launch_bounds__(128)
k_col_views(int cnt, const uint32_t* __restrict__ tile_nnz_ptr, const uint16_t* __restrict__ masks_t,
            const uint8_t* __restrict__ rc_idx, const T* __restrict__ vals,
            uint32_t* __restrict__ col_rec, T* __restrict__ vals_t)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= cnt) return;
    const uint4* m4 = reinterpret_cast<const uint4*>(masks_t + (size_t)t * 16);
    const uint4 a = m4[0], b = m4[1];
    const unsigned w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    unsigned rec[16];
    unsigned run = 0;
#pragma unroll
    for (int c = 0; c < 16; ++c) {
        const unsigned m = (w[c >> 1] >> ((c & 1) * 16)) & 0xFFFFu;
        rec[c] = m | (run << 24);       // offset in the top byte: disjoint from the row records' byte (bits 16-23), see step3.cu
        run += __popc(m);
    }
    uint4* out = reinterpret_cast<uint4*>(col_rec + (size_t)t * 16);
    out[0] = make_uint4(rec[0], rec[1], rec[2], rec[3]);
    out[1] = make_uint4(rec[4], rec[5], rec[6], rec[7]);
    out[2] = make_uint4(rec[8], rec[9], rec[10], rec[11]);
    out[3] = make_uint4(rec[12], rec[13], rec[14], rec[15]);
    const uint32_t s = tile_nnz_ptr[t], e = tile_nnz_ptr[t + 1];
    const uint32_t* my = col_rec + (size_t)t * 16;      // just written by this thread
    for (uint32_t x = s; x < e; ++x) {
        const unsigned rc = rc_idx[x];
        const unsigned r = rc >> 4, c = rc & 15u;
        const unsigned cr = my[c];
        vals_t[pem_col_slot(s, cr, r)] = vals[x];
    }
}

// ---- value refresh (pem_tiled_set_values) -----------------------------------------------------------
// vals[x] = V[pos[x]], and the same value into vals_t when the step-3 view exists (pem_write_slots)
template <class T>
__global__ void __launch_bounds__(256)
k_refresh_vals(int cnt, const uint32_t* __restrict__ tile_nnz_ptr, const uint32_t* __restrict__ pos,
               const T* __restrict__ V, const uint8_t* __restrict__ rc_idx, const uint32_t* __restrict__ col_rec,
               T* __restrict__ vals, T* __restrict__ vals_t)
{
    pem_write_slots((int64_t)blockIdx.x * blockDim.x + threadIdx.x, threadIdx.x, cnt, tile_nnz_ptr, rc_idx, col_rec, vals,
                    vals_t, [=](uint32_t x, int64_t) { return V[pos[x]]; });
}
// V in slot order, no map: pem_tiled_refresh_from_result, whose source result holds its values in the handle's slots
template <class T>
__global__ void __launch_bounds__(256)
k_refresh_slots(int cnt, const uint32_t* __restrict__ tile_nnz_ptr, const T* __restrict__ V,
                const uint8_t* __restrict__ rc_idx, const uint32_t* __restrict__ col_rec, T* __restrict__ vals,
                T* __restrict__ vals_t)
{
    pem_write_slots((int64_t)blockIdx.x * blockDim.x + threadIdx.x, threadIdx.x, cnt, tile_nnz_ptr, rc_idx, col_rec, vals,
                    vals_t, [=](uint32_t x, int64_t) { return V[x]; });
}

// tile products of one A tile, at tile level (length of B's tile row) and through B's row slices;
// the smaller of the two is what step 1 will expand.  Summed per tile row.
__global__ void __launch_bounds__(256)
k_tile_prodcost(const uint16_t* __restrict__ col_occ, const int32_t* __restrict__ tile_row,
                const int32_t* __restrict__ tile_col, int cnt, const int32_t* __restrict__ Brp,
                const int64_t* __restrict__ srow_ptr, unsigned long long* __restrict__ row_tile_cost,
                unsigned long long* __restrict__ row_sliced_cost)
{
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= cnt) return;
    const int k = tile_col[t];
    const unsigned long long pt = (unsigned long long)(Brp[k + 1] - Brp[k]);
    unsigned occ = col_occ[t];
    const int64_t* sp = srow_ptr + (size_t)k * 16;
    unsigned long long ps = 0;
    while (occ) {
        const int c = __ffs(occ) - 1;
        occ &= occ - 1;
        ps += (unsigned long long)(sp[c + 1] - sp[c]);
    }
    if (pt) atomicAdd(&row_tile_cost[tile_row[t]], pt);
    if (ps) atomicAdd(&row_sliced_cost[tile_row[t]], ps);
}

// ---- transpose of a tiled matrix on the device ----------------------------------------------------
__global__ void __launch_bounds__(256)
k_transpose_keys(const int32_t* __restrict__ tile_row, const int32_t* __restrict__ tile_col, int cnt, int rbits,
                 uint64_t* __restrict__ keys, int32_t* __restrict__ ids)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= cnt) return;
    keys[t] = ((uint64_t)(unsigned)tile_col[t] << rbits) | (uint64_t)(unsigned)tile_row[t];   // new (row, col)
    ids[t] = t;
}

__global__ void __launch_bounds__(256)
k_transpose_counts(const int32_t* __restrict__ perm, const uint32_t* __restrict__ nnz_ptr, int cnt, int64_t* __restrict__ out)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t > cnt) return;
    out[t] = t < cnt ? (int64_t)(nnz_ptr[perm[t] + 1] - nnz_ptr[perm[t]]) : 0;
}

// thread per tile of the transpose: masks swap roles, values (and their value-map entries) move to their column-major
// position
template <class T>
__global__ void __launch_bounds__(128)
k_transpose_tiles(int cnt, int tile_rows_new, const int32_t* __restrict__ perm, const int64_t* __restrict__ new_ptr,
                  const uint32_t* __restrict__ o_nnz_ptr, const uint16_t* __restrict__ o_masks,
                  const uint16_t* __restrict__ o_masks_t, const int32_t* __restrict__ o_row, const int32_t* __restrict__ o_col,
                  const uint16_t* __restrict__ o_col_occ, const uint16_t* __restrict__ o_row_occ,
                  const uint8_t* __restrict__ o_rc, const T* __restrict__ o_vals, const uint32_t* __restrict__ o_pos,
                  uint32_t* __restrict__ n_nnz_ptr, uint16_t* __restrict__ n_masks, uint16_t* __restrict__ n_masks_t,
                  uint8_t* __restrict__ n_row_ptr, int32_t* __restrict__ n_row, int32_t* __restrict__ n_col,
                  int32_t* __restrict__ n_tile_row_ptr, uint16_t* __restrict__ n_col_occ, uint16_t* __restrict__ n_row_occ,
                  uint8_t* __restrict__ n_rc, T* __restrict__ n_vals, uint32_t* __restrict__ n_pos)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= cnt) return;
    const int o = perm[t];
    const uint4* mt4 = reinterpret_cast<const uint4*>(o_masks_t + (size_t)o * 16);     // new row masks
    const uint4 a = mt4[0], b = mt4[1];
    const uint4* m4 = reinterpret_cast<const uint4*>(o_masks + (size_t)o * 16);        // new column masks
    reinterpret_cast<uint4*>(n_masks + (size_t)t * 16)[0] = a;
    reinterpret_cast<uint4*>(n_masks + (size_t)t * 16)[1] = b;
    reinterpret_cast<uint4*>(n_masks_t + (size_t)t * 16)[0] = m4[0];
    reinterpret_cast<uint4*>(n_masks_t + (size_t)t * 16)[1] = m4[1];
    const unsigned w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    unsigned rp[16], packed[4] = {0, 0, 0, 0};
    unsigned run = 0;
#pragma unroll
    for (int r = 0; r < 16; ++r) {
        rp[r] = run;
        packed[r >> 2] |= run << (8 * (r & 3));
        run += __popc((w[r >> 1] >> ((r & 1) * 16)) & 0xFFFFu);
    }
    *reinterpret_cast<uint4*>(n_row_ptr + (size_t)t * 16) = make_uint4(packed[0], packed[1], packed[2], packed[3]);
    const int nr = o_col[o], nc = o_row[o];
    n_row[t] = nr;
    n_col[t] = nc;
    n_col_occ[t] = o_row_occ[o];
    n_row_occ[t] = o_col_occ[o];
    const uint32_t ns = (uint32_t)new_ptr[t];
    n_nnz_ptr[t] = ns;
    const int prev = t ? o_col[perm[t - 1]] : -1;
    for (int r = prev + 1; r <= nr; ++r) n_tile_row_ptr[r] = t;
    if (t == cnt - 1) {
        for (int r = nr + 1; r <= tile_rows_new; ++r) n_tile_row_ptr[r] = cnt;
        n_nnz_ptr[cnt] = (uint32_t)new_ptr[cnt];
    }
    const uint32_t s = o_nnz_ptr[o], e = o_nnz_ptr[o + 1];
    for (uint32_t x = s; x < e; ++x) {
        const unsigned rc = o_rc[x];
        const unsigned r = rc >> 4, c = rc & 15u;          // old (r, c) -> new (c, r)
        unsigned first = 0, m = 0;                          // rp[c], new row mask c (dynamic c: selects)
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            first = c == (unsigned)j ? rp[j] : first;
            m = c == (unsigned)j ? ((w[j >> 1] >> ((j & 1) * 16)) & 0xFFFFu) : m;
        }
        const uint32_t at = ns + first + __popc(m & ((1u << r) - 1u));
        n_vals[at] = o_vals[x];
        n_pos[at] = o_pos[x];
        n_rc[at] = (uint8_t)((c << 4) | r);
    }
}

bool is_device_ptr(const void* p)
{
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        (void)cudaGetLastError();
        return false;
    }
    return at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
}

int tile_row_flops(pem_ctx* ctx, const pem_tiled* A, const pem_tiled* B, unsigned long long** d_out)
{
    uint32_t* b_row_nnz = nullptr;
    unsigned long long* trf = nullptr;     // handed to the caller on success
    pem_guard g(ctx, b_row_nnz, trf);
    PEM_TRY(pem_alloc(ctx, &b_row_nnz, (size_t)B->tile_rows * 16));
    PEM_TRY(pem_alloc(ctx, &trf, (size_t)A->tile_rows));
    PEM_CK(cudaMemsetAsync(b_row_nnz, 0, (size_t)(B->tile_rows ? B->tile_rows : 1) * 16 * 4, ctx->stream));
    PEM_CK(cudaMemsetAsync(trf, 0, (size_t)(A->tile_rows ? A->tile_rows : 1) * 8, ctx->stream));
    if (B->tiles) {
        k_row_nnz<<<pem_div_up(B->tiles, 256), 256, 0, ctx->stream>>>(B->masks, B->tile_row_idx, B->tiles, b_row_nnz);
        PEM_LAUNCHED();
    }
    if (A->tiles) {
        k_tile_flop<<<pem_div_up(A->tiles, 256), 256, 0, ctx->stream>>>(A->masks_t, A->tile_row_idx, A->tile_col_idx,
                                                                        A->tiles, b_row_nnz, B->rows, trf);
        PEM_LAUNCHED();
    }
    pem_free(ctx, b_row_nnz);
    *d_out = std::exchange(trf, nullptr);
    return PEM_OK;
}

}  // namespace

// COO -> tiled CSR for either value type (V points at doubles or floats according to dtype)
static int convert_coo_any(pem_ctx* ctx, int32_t rows, int32_t cols, int64_t nnz,
                           const int32_t* I, const int32_t* J, const void* V, int dtype, int transpose,
                           pem_tiled** out, pem_times* times)
{
    PEM_RANGE("pem_convert_coo");
    const size_t vsz = pem_vsize(dtype);
    if (!ctx || !out) return PEM_ERR_ARG;
    *out = nullptr;
    if (rows < 0 || cols < 0 || nnz < 0) return ctx->fail(PEM_ERR_ARG, "negative size");
    if (nnz > 0 && (!I || !J || !V)) return ctx->fail(PEM_ERR_ARG, "null COO array");
    if (nnz >= (int64_t(1) << 32) - 1) return ctx->fail(PEM_ERR_LIMIT, "nnz must be below 2^32-1 (32-bit tile value offsets)");
    PEM_CK(cudaSetDevice(ctx->device));
    auto wall0 = std::chrono::high_resolution_clock::now();
    if (transpose) { int32_t t = rows; rows = cols; cols = t; }

    pem_tiled_ptr T = pem_tiled_new(ctx, dtype, rows, cols, nnz);
    int32_t *sI = nullptr, *sJ = nullptr;      // device copies of a COO that came from the host
    char* sV = nullptr;
    uint64_t *keys = nullptr, *keys_sorted = nullptr;
    uint32_t *pos = nullptr, *start_tmp = nullptr;
    char* tmp = nullptr;
    pem_guard g(ctx, sI, sJ, sV, keys, keys_sorted, pos, start_tmp, tmp);
    // on failure nothing may still be writing a buffer that goes back to the cache (the copy stream may still be
    // filling sV or reading T->val_pos): declared after T and the guard, so it waits before either frees
    struct wait_on_failure {
        pem_ctx* ctx;
        pem_tiled** out;
        ~wait_on_failure()
        {
            if (*out) return;
            cudaStreamSynchronize(ctx->copy_stream);
            cudaStreamSynchronize(ctx->stream);
        }
    } idle{ctx, out};

    float kernel_ms = 0.f;

    if (nnz > 0) {
        int cb = h_bits_for(T->tile_cols), rb = h_bits_for(T->tile_rows);
        // stage the COO on the device if it came from the host (pinned or pageable)
        const bool own = !is_device_ptr(I);
        if (own) {
            PEM_TRY(pem_alloc(ctx, &sI, (size_t)nnz));
            PEM_TRY(pem_alloc(ctx, &sJ, (size_t)nnz));
            PEM_TRY(pem_alloc(ctx, &sV, (size_t)nnz * vsz));
            PEM_CK(cudaMemcpyAsync(sI, I, (size_t)nnz * 4, cudaMemcpyHostToDevice, ctx->stream));
            PEM_CK(cudaMemcpyAsync(sJ, J, (size_t)nnz * 4, cudaMemcpyHostToDevice, ctx->stream));
            // the values travel on a second stream, behind the coordinates and under key generation + sort
            PEM_CK(cudaEventRecord(ctx->ev_copy[0], ctx->stream));
            PEM_CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_copy[0], 0));
            PEM_CK(cudaMemcpyAsync(sV, V, (size_t)nnz * vsz, cudaMemcpyHostToDevice, ctx->copy_stream));
            PEM_CK(cudaEventRecord(ctx->ev_copy[1], ctx->copy_stream));
        }
        const int32_t* dI = own ? sI : I;
        const int32_t* dJ = own ? sJ : J;
        const char* dV = own ? sV : static_cast<const char*>(V);
        PEM_TRY(pem_alloc(ctx, &keys, (size_t)nnz));
        PEM_TRY(pem_alloc(ctx, &keys_sorted, (size_t)nnz));
        PEM_TRY(pem_alloc(ctx, &pos, (size_t)nnz));
        // the sorted positions are the value map: slot x of vals holds V[val_pos[x]] (pem_tiled_set_values)
        PEM_TRY(pem_tiled_alloc_values(ctx, T.get()));
        PEM_CK(cudaMemsetAsync(ctx->d_scalars, 0, PEM_NSCALARS * sizeof(int64_t), ctx->stream));

        int grid = (int)std::min<int64_t>(pem_div_up(nnz, 256), (int64_t)ctx->sm_count * 32);
        k_make_keys<<<grid, 256, 0, ctx->stream>>>(dI, dJ, nnz, rows, cols, transpose, cb, keys, pos, ctx->d_scalars);
        PEM_LAUNCHED();

        // one radix sort of (key, original position) over the bits in use
        size_t tmp_bytes = 0, tmp2 = 0;
        PEM_CK(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, keys, keys_sorted, pos, T->val_pos, nnz, 0, 8 + cb + rb, ctx->stream));
        PEM_TRY(pem_alloc(ctx, &start_tmp, (size_t)nnz + 1));
        cub::CountingInputIterator<uint32_t> iota(0);
        HeadPred pred{keys_sorted};
        int64_t* d_count = ctx->d_scalars + SC_COUNT;
        PEM_CK(cub::DeviceSelect::If(nullptr, tmp2, iota, start_tmp, d_count, nnz, pred, ctx->stream));
        PEM_TRY(pem_alloc(ctx, &tmp, std::max(tmp_bytes, tmp2)));
        PEM_CK(cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, keys, keys_sorted, pos, T->val_pos, nnz, 0, 8 + cb + rb, ctx->stream));
        PEM_CK(cub::DeviceSelect::If(tmp, tmp2, iota, start_tmp, d_count, nnz, pred, ctx->stream));
        k_rc_idx<<<pem_div_up(nnz, 256), 256, 0, ctx->stream>>>(keys_sorted, nnz, T->rc_idx);
        PEM_LAUNCHED();
        cudaStream_t gather = ctx->stream;
        if (own) {
            // The values are gathered into tile order on the COPY stream, behind their upload; the engine's
            // stream does not wait here: tile build and the symbolic steps of a product need masks only, so
            // they run underneath the upload.  pem_tiled_wait_vals joins the two streams for the first reader.
            PEM_CK(cudaEventCreateWithFlags(&T->ev_vals, cudaEventDisableTiming));
            PEM_CK(cudaEventRecord(ctx->ev_copy[0], ctx->stream));                  // sorted positions are final
            PEM_CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_copy[0], 0));
            gather = ctx->copy_stream;
        }
        pem_by_dtype(dtype, [&](auto v) {
            using VT = decltype(v);
            k_gather_vals<VT><<<pem_div_up(nnz, 256), 256, 0, gather>>>(T->val_pos, pem_vals<VT>(dV), nnz, pem_vals<VT>(T->vals));
        });
        PEM_LAUNCHED();
        if (own) {
            PEM_CK(cudaEventRecord(T->ev_vals, ctx->copy_stream));
            T->vals_pending = true;
            T->pend_buf = std::exchange(sV, nullptr);                             // freed once the gather is known to be done
        }
        pem_free(ctx, pos);
        PEM_CK(cudaMemcpyAsync(ctx->h_scalars, ctx->d_scalars, PEM_NSCALARS * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
        PEM_CK(cudaStreamSynchronize(ctx->stream));
        pem_free(ctx, tmp);
        pem_free(ctx, keys);
        pem_free(ctx, sI);
        pem_free(ctx, sJ);
        // default contract: the caller's arrays are free again when this call returns, so the host waits for the
        // values' upload (not for their gather); PEM_OPT_ASYNC_VALUES hands that wait to the caller
        if (own && !ctx->opt_async_vals) PEM_CK(cudaEventSynchronize(ctx->ev_copy[1]));
        if (ctx->h_scalars[SC_ERR] & 1) return ctx->fail(PEM_ERR_RANGE, "COO coordinate outside the matrix");
        int64_t cnt = ctx->h_scalars[SC_COUNT];
        if (cnt >= (int64_t(1) << 31) - 1) return ctx->fail(PEM_ERR_LIMIT, "more than 2^31 tiles");
        T->tiles = (int32_t)cnt;
        PEM_TRY(pem_tiled_alloc_tiles(ctx, T.get()));
        PEM_CK(cudaMemcpyAsync(T->tile_nnz_ptr, start_tmp, (size_t)cnt * 4, cudaMemcpyDeviceToDevice, ctx->stream));
        pem_free(ctx, start_tmp);
        PEM_CK(cudaEventRecord(ctx->ev[0], ctx->stream));
        k_build_tiles<<<pem_div_up(cnt, 128), 128, 0, ctx->stream>>>(
            keys_sorted, T->tile_nnz_ptr, (int)cnt, (uint32_t)nnz, cb, T->tile_rows, T->masks, T->masks_t,
            T->row_ptr, T->tile_col_idx, T->tile_row_idx, T->tile_row_ptr, T->col_occ, T->row_occ, ctx->d_scalars);
        PEM_LAUNCHED();
        PEM_CK(cudaEventRecord(ctx->ev[1], ctx->stream));
        PEM_CK(cudaMemcpyAsync(ctx->h_scalars, ctx->d_scalars, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
        PEM_TRY(pem_tiled_publish(ctx, T.get()));
        pem_free(ctx, keys_sorted);
        if (ctx->h_scalars[SC_ERR] & 2) return ctx->fail(PEM_ERR_DUPLICATE, "duplicate (i,j) in the COO input");
        cudaEventElapsedTime(&kernel_ms, ctx->ev[0], ctx->ev[1]);
    } else {
        PEM_TRY(pem_tiled_alloc(ctx, T.get()));
        PEM_CK(cudaMemsetAsync(T->tile_row_ptr, 0, ((size_t)T->tile_rows + 1) * 4, ctx->stream));
        PEM_CK(cudaMemsetAsync(T->tile_nnz_ptr, 0, 4, ctx->stream));
        PEM_TRY(pem_tiled_publish(ctx, T.get()));
    }
    if (times) {
        auto wall1 = std::chrono::high_resolution_clock::now();
        times->convert_kernel_ms = kernel_ms;
        times->convert_total_ms = std::chrono::duration<double, std::milli>(wall1 - wall0).count();
    }
    *out = T.release();
    return PEM_OK;
}

extern "C" {

int pem_convert_coo(pem_ctx* ctx, int32_t rows, int32_t cols, int64_t nnz,
                    const int32_t* I, const int32_t* J, const double* V, int transpose,
                    pem_tiled** out, pem_times* times)
{
    return convert_coo_any(ctx, rows, cols, nnz, I, J, V, PEM_F64, transpose, out, times);
}

int pem_convert_coo_f32(pem_ctx* ctx, int32_t rows, int32_t cols, int64_t nnz,
                        const int32_t* I, const int32_t* J, const float* V, int transpose,
                        pem_tiled** out, pem_times* times)
{
    return convert_coo_any(ctx, rows, cols, nnz, I, J, V, PEM_F32, transpose, out, times);
}

int pem_convert_csr(pem_ctx* ctx, int32_t rows, int32_t cols, const int32_t* row_ptr, const int32_t* col_idx,
                    const double* vals, int transpose, pem_tiled** out, pem_times* times)
{
    PEM_RANGE("pem_convert_csr");
    if (!ctx || !out) return PEM_ERR_ARG;
    *out = nullptr;
    if (rows < 0 || cols < 0 || !row_ptr) return ctx->fail(PEM_ERR_ARG, "bad CSR arguments");
    PEM_CK(cudaSetDevice(ctx->device));
    auto wall0 = std::chrono::high_resolution_clock::now();
    const bool on_device = is_device_ptr(row_ptr);
    int32_t first = 0, last = 0;
    if (on_device) {
        PEM_CK(cudaMemcpyAsync(&first, row_ptr, 4, cudaMemcpyDeviceToHost, ctx->stream));
        PEM_CK(cudaMemcpyAsync(&last, row_ptr + rows, 4, cudaMemcpyDeviceToHost, ctx->stream));
        PEM_CK(cudaStreamSynchronize(ctx->stream));
    } else {
        first = row_ptr[0]; last = row_ptr[rows];
    }
    if (first != 0 || last < 0) return ctx->fail(PEM_ERR_ARG, "CSR row pointer must start at 0 and be non-negative");
    const int64_t nnz = last;
    if (nnz > 0 && (!col_idx || !vals)) return ctx->fail(PEM_ERR_ARG, "null CSR array");
    // everything onto the device (the row pointer expands to one row index per nonzero there), then the COO path
    int32_t *d_rp = nullptr, *dI = nullptr, *dJ = nullptr;
    double* dV = nullptr;
    pem_guard g(ctx, dI, d_rp, dJ, dV);
    PEM_TRY(pem_alloc(ctx, &dI, (size_t)nnz));
    const int32_t* rp = row_ptr;
    const int32_t* J = col_idx;
    const double* V = vals;
    if (!on_device) {
        PEM_TRY(pem_alloc(ctx, &d_rp, (size_t)rows + 1));
        PEM_TRY(pem_alloc(ctx, &dJ, (size_t)nnz));
        PEM_TRY(pem_alloc(ctx, &dV, (size_t)nnz));
        PEM_CK(cudaMemcpyAsync(d_rp, row_ptr, ((size_t)rows + 1) * 4, cudaMemcpyHostToDevice, ctx->stream));
        if (nnz) PEM_CK(cudaMemcpyAsync(dJ, col_idx, (size_t)nnz * 4, cudaMemcpyHostToDevice, ctx->stream));
        if (nnz) PEM_CK(cudaMemcpyAsync(dV, vals, (size_t)nnz * 8, cudaMemcpyHostToDevice, ctx->stream));
        rp = d_rp; J = dJ; V = dV;
    }
    if (nnz > 0) {
        k_csr_rows<<<pem_div_up(nnz, 256), 256, 0, ctx->stream>>>(rp, rows, nnz, dI);
        PEM_LAUNCHED();
    }
    PEM_TRY(pem_convert_coo(ctx, rows, cols, nnz, dI, J, V, transpose, out, times));
    if (times)
        times->convert_total_ms = std::chrono::duration<double, std::milli>(std::chrono::high_resolution_clock::now() - wall0).count();
    return PEM_OK;
}

}  // extern "C"

// Join the engine's stream with the upload + gather of a freshly converted operand's values (see
// pem_convert_coo); a no-op for every later call.
int pem_tiled_wait_vals(pem_ctx* ctx, const pem_tiled* Tc)
{
    pem_tiled* T = const_cast<pem_tiled*>(Tc);
    if (!T->vals_pending) return PEM_OK;
    PEM_CK(cudaStreamWaitEvent(ctx->stream, T->ev_vals, 0));
    // the staging buffers go back to the cache in the engine's stream order, i.e. behind the wait above
    if (T->pend_buf) pem_free_bytes(ctx, T->pend_buf);
    T->pend_buf = nullptr;
    T->vals_pending = false;
    return PEM_OK;
}

// Row slices of a tiled matrix, built once and cached on the handle (the handle is logically
// const for the caller; the cache is the one mutable part).
int pem_tiled_build_srow(pem_ctx* ctx, const pem_tiled* Bc)
{
    pem_tiled* B = const_cast<pem_tiled*>(Bc);
    if (B->srow_ptr) return PEM_OK;
    // a handle's caches outlive any product: never built from a graph's arena (the capture is given up instead)
    if (ctx->cap) return ctx->fail(PEM_ERR_CUDA, "operand cache built inside a graph capture");
    const size_t rows16 = (size_t)B->tile_rows * 16;
    int64_t* ptr = nullptr;
    int32_t* tl = nullptr;
    unsigned* cursor = nullptr;
    pem_guard g(ctx, ptr, tl, cursor);
    PEM_TRY(pem_alloc(ctx, &ptr, rows16 + 1));
    PEM_CK(cudaMemsetAsync(ptr, 0, (rows16 + 1) * 8, ctx->stream));
    if (B->tiles) {
        k_srow_count<<<pem_div_up(B->tiles, 256), 256, 0, ctx->stream>>>(B->row_occ, B->tile_row_idx, B->tiles,
                                                                         (unsigned long long*)ptr);
        PEM_LAUNCHED();
    }
    PEM_TRY(pem_scan_exclusive_i64(ctx, ptr, (int64_t)rows16 + 1));
    PEM_CK(cudaMemcpyAsync(ctx->h_scalars, ptr + rows16, 8, cudaMemcpyDeviceToHost, ctx->stream));
    PEM_CK(cudaStreamSynchronize(ctx->stream));
    const int64_t total = ctx->h_scalars[0];
    PEM_TRY(pem_alloc(ctx, &tl, (size_t)total));
    if (B->tiles) {
        PEM_TRY(pem_alloc(ctx, &cursor, rows16));
        PEM_CK(cudaMemsetAsync(cursor, 0, rows16 * 4, ctx->stream));
        k_srow_fill<<<pem_div_up(B->tiles, 256), 256, 0, ctx->stream>>>(B->row_occ, B->tile_row_idx, B->tiles, ptr, cursor, tl);
        PEM_LAUNCHED();
        pem_free(ctx, cursor);
    }
    B->srow_ptr = std::exchange(ptr, nullptr);
    B->srow_total = total;
    B->srow_tile = std::exchange(tl, nullptr);
    return PEM_OK;
}

// Step-3 views of a tiled matrix, built once per role and cached on the handle.
int pem_tiled_build_views(pem_ctx* ctx, const pem_tiled* Tc, bool as_a, bool as_b)
{
    pem_tiled* T = const_cast<pem_tiled*>(Tc);
    const size_t n16 = (size_t)T->tiles * 16;
    if (ctx->cap && ((as_a && !T->row_rec) || (as_b && !T->col_rec)))
        return ctx->fail(PEM_ERR_CUDA, "operand cache built inside a graph capture");
    if (as_a && !T->row_rec) {
        uint32_t* rec = nullptr;
        pem_guard g(ctx, rec);
        PEM_TRY(pem_alloc(ctx, &rec, n16));
        if (n16) {
            k_row_rec<<<pem_div_up((int64_t)n16, 256), 256, 0, ctx->stream>>>(T->masks, T->row_ptr, (int64_t)n16, rec);
            PEM_LAUNCHED();
        }
        T->row_rec = std::exchange(rec, nullptr);
    }
    if (as_b && !T->col_rec) {
        PEM_TRY(pem_tiled_wait_vals(ctx, T));
        uint32_t* rec = nullptr;
        double* vt = nullptr;
        pem_guard g(ctx, rec, vt);
        PEM_TRY(pem_alloc(ctx, &rec, n16));
        PEM_TRY(pem_alloc_bytes(ctx, (void**)&vt, std::max<size_t>(1, (size_t)T->nnz * pem_vsize(T->dtype))));
        if (T->tiles) {
            pem_by_dtype(T->dtype, [&](auto v) {
                using VT = decltype(v);
                k_col_views<VT><<<pem_div_up(T->tiles, 128), 128, 0, ctx->stream>>>(
                    T->tiles, T->tile_nnz_ptr, T->masks_t, T->rc_idx, pem_vals<VT>(T->vals), rec, pem_vals<VT>(vt));
            });
            PEM_LAUNCHED();
        }
        T->col_rec = std::exchange(rec, nullptr);
        T->vals_t = std::exchange(vt, nullptr);
    }
    return PEM_OK;
}

// new values on an existing pattern, in place (pem_tiled_set_values / _f32)
static int set_values_any(pem_ctx* ctx, pem_tiled* T, const void* V, int dtype)
{
    PEM_RANGE("pem_tiled_set_values");
    if (!ctx || !T) return PEM_ERR_ARG;
    if (T->dtype != dtype)
        return ctx->fail(PEM_ERR_ARG, T->dtype == PEM_F32 ? "fp32 matrix: refresh its values with pem_tiled_set_values_f32"
                                                          : "fp64 matrix: refresh its values with pem_tiled_set_values");
    if (T->nnz == 0) return PEM_OK;
    if (!V) return ctx->fail(PEM_ERR_ARG, "null value array");
    PEM_CK(cudaSetDevice(ctx->device));
    PEM_TRY(pem_tiled_wait_vals(ctx, T));           // a gather still running on the copy stream would overwrite the new values
    const size_t bytes = (size_t)T->nnz * pem_vsize(dtype);
    char* staged = nullptr;
    pem_guard g(ctx, staged);
    const void* dV = V;
    if (!is_device_ptr(V)) {
        PEM_TRY(pem_alloc_bytes(ctx, (void**)&staged, bytes));
        PEM_CK(cudaMemcpyAsync(staged, V, bytes, cudaMemcpyHostToDevice, ctx->stream));
        PEM_CK(cudaEventRecord(ctx->ev_copy[1], ctx->stream));
        dV = staged;
    }
    if (T->tiles) {
        pem_by_dtype(dtype, [&](auto v) {
            using VT = decltype(v);
            k_refresh_vals<VT><<<pem_div_up(T->tiles, 256), 256, 0, ctx->stream>>>(
                T->tiles, T->tile_nnz_ptr, T->val_pos, pem_vals<VT>(dV), T->rc_idx, T->col_rec, pem_vals<VT>(T->vals),
                pem_vals<VT>(T->vals_t));
        });
        PEM_LAUNCHED();
    }
    // default contract, as for conversion: a host V is free again when the call returns (the kernel may still run)
    if (staged) PEM_CK(cudaEventSynchronize(ctx->ev_copy[1]));
    return PEM_OK;
}

// new values already in T's slot order (device array of T->nnz values of T's dtype), in place: a copy into vals, or,
// when the column-major view exists, one pass that writes vals and vals_t
int pem_tiled_write_slots(pem_ctx* ctx, pem_tiled* T, const void* dV)
{
    if (T->nnz == 0) return PEM_OK;
    if (!T->vals_t) {
        PEM_CK(cudaMemcpyAsync(T->vals, dV, (size_t)T->nnz * pem_vsize(T->dtype), cudaMemcpyDeviceToDevice, ctx->stream));
        return PEM_OK;
    }
    pem_by_dtype(T->dtype, [&](auto v) {
        using VT = decltype(v);
        k_refresh_slots<VT><<<pem_div_up(T->tiles, 256), 256, 0, ctx->stream>>>(
            T->tiles, T->tile_nnz_ptr, pem_vals<VT>(dV), T->rc_idx, T->col_rec, pem_vals<VT>(T->vals), pem_vals<VT>(T->vals_t));
    });
    PEM_LAUNCHED();
    return PEM_OK;
}

extern "C" {

int pem_tiled_set_values(pem_ctx* ctx, pem_tiled* t, const double* V) { return set_values_any(ctx, t, V, PEM_F64); }

int pem_tiled_set_values_f32(pem_ctx* ctx, pem_tiled* t, const float* V) { return set_values_any(ctx, t, V, PEM_F32); }

int pem_tiled_transpose(pem_ctx* ctx, const pem_tiled* A, pem_tiled** out)
{
    PEM_RANGE("pem_tiled_transpose");
    if (!ctx || !A || !out) return PEM_ERR_ARG;
    *out = nullptr;
    PEM_CK(cudaSetDevice(ctx->device));
    PEM_TRY(pem_tiled_wait_vals(ctx, A));
    pem_tiled_ptr T = pem_tiled_new(ctx, A->dtype, A->cols, A->rows, A->nnz);
    T->tiles = A->tiles;
    const size_t n = (size_t)A->tiles;
    uint64_t *keys = nullptr, *keys2 = nullptr;
    int32_t *ids = nullptr, *perm = nullptr;
    int64_t* nptr = nullptr;
    char* tmp = nullptr;
    pem_guard g(ctx, keys, keys2, ids, perm, nptr, tmp);
    PEM_TRY(pem_tiled_alloc(ctx, T.get()));
    if (n == 0) {
        PEM_CK(cudaMemsetAsync(T->tile_row_ptr, 0, ((size_t)T->tile_rows + 1) * 4, ctx->stream));
        PEM_CK(cudaMemsetAsync(T->tile_nnz_ptr, 0, 4, ctx->stream));
        PEM_TRY(pem_tiled_publish(ctx, T.get()));
        *out = T.release();
        return PEM_OK;
    }
    const int rbits = h_bits_for(A->tile_rows), cbits = h_bits_for(A->tile_cols);
    PEM_TRY(pem_alloc(ctx, &keys, n)); PEM_TRY(pem_alloc(ctx, &keys2, n));
    PEM_TRY(pem_alloc(ctx, &ids, n)); PEM_TRY(pem_alloc(ctx, &perm, n));
    PEM_TRY(pem_alloc(ctx, &nptr, n + 1));
    k_transpose_keys<<<pem_div_up((int64_t)n, 256), 256, 0, ctx->stream>>>(A->tile_row_idx, A->tile_col_idx, (int)n, rbits, keys, ids);
    PEM_LAUNCHED();
    size_t tb = 0;
    PEM_CK(cub::DeviceRadixSort::SortPairs(nullptr, tb, keys, keys2, ids, perm, (int64_t)n, 0, rbits + cbits, ctx->stream));
    PEM_TRY(pem_alloc(ctx, &tmp, tb));
    PEM_CK(cub::DeviceRadixSort::SortPairs(tmp, tb, keys, keys2, ids, perm, (int64_t)n, 0, rbits + cbits, ctx->stream));
    ctx->launches += 2 + (rbits + cbits + 7) / 8;
    k_transpose_counts<<<pem_div_up((int64_t)n + 1, 256), 256, 0, ctx->stream>>>(perm, A->tile_nnz_ptr, (int)n, nptr);
    PEM_LAUNCHED();
    PEM_TRY(pem_scan_exclusive_i64(ctx, nptr, (int64_t)n + 1));
    pem_by_dtype(A->dtype, [&](auto v) {
        using VT = decltype(v);
        k_transpose_tiles<VT><<<pem_div_up((int64_t)n, 128), 128, 0, ctx->stream>>>(
            (int)n, T->tile_rows, perm, nptr, A->tile_nnz_ptr, A->masks, A->masks_t, A->tile_row_idx, A->tile_col_idx, A->col_occ,
            A->row_occ, A->rc_idx, pem_vals<VT>(A->vals), A->val_pos, T->tile_nnz_ptr, T->masks, T->masks_t, T->row_ptr,
            T->tile_row_idx, T->tile_col_idx, T->tile_row_ptr, T->col_occ, T->row_occ, T->rc_idx, pem_vals<VT>(T->vals),
            T->val_pos);
    });
    PEM_LAUNCHED();
    PEM_TRY(pem_tiled_publish(ctx, T.get()));
    pem_free(ctx, keys); pem_free(ctx, keys2); pem_free(ctx, ids); pem_free(ctx, perm); pem_free(ctx, nptr); pem_free(ctx, tmp);
    *out = T.release();
    return PEM_OK;
}

int pem_count_flop(pem_ctx* ctx, const pem_tiled* A, const pem_tiled* B, uint64_t* flop)
{
    if (!ctx || !A || !B || !flop) return PEM_ERR_ARG;
    if (A->cols != B->rows) return ctx->fail(PEM_ERR_ARG, "inner dimensions differ");
    PEM_CK(cudaSetDevice(ctx->device));
    unsigned long long* trf = nullptr;
    pem_guard g(ctx, trf);
    PEM_TRY(tile_row_flops(ctx, A, B, &trf));
    std::vector<unsigned long long> h((size_t)A->tile_rows);
    if (A->tile_rows) PEM_CK(cudaMemcpyAsync(h.data(), trf, h.size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
    PEM_CK(cudaStreamSynchronize(ctx->stream));
    pem_free(ctx, trf);
    uint64_t f = 0;
    for (auto v : h) f += v;
    *flop = f;
    return PEM_OK;
}

int pem_partition_panels(pem_ctx* ctx, const pem_tiled* A, const pem_tiled* B, int nparts, int32_t* bounds)
{
    if (!ctx || !A || !B || !bounds || nparts <= 0) return PEM_ERR_ARG;
    if (A->cols != B->rows) return ctx->fail(PEM_ERR_ARG, "inner dimensions differ");
    PEM_CK(cudaSetDevice(ctx->device));
    const size_t ntr = (size_t)A->tile_rows;
    unsigned long long *trf = nullptr, *cp = nullptr, *cs = nullptr;
    pem_guard g(ctx, trf, cp, cs);
    PEM_TRY(tile_row_flops(ctx, A, B, &trf));
    std::vector<unsigned long long> h(ntr), hp(ntr, 0), hs(ntr, 0);
    if (ntr) PEM_CK(cudaMemcpyAsync(h.data(), trf, ntr * 8, cudaMemcpyDeviceToHost, ctx->stream));
    // Weight of a tile row = its flop (the reference's and the north star's measure, spgemm.cu:1068-1079)
    // + 16 x the tile products step 1 will expand for it: steps 1 and 2 and the per-pair part of step 3
    // cost per tile PAIR, not per flop, and on power-law inputs the two are distributed very differently
    // (hub rows: many flops in few tiles; ordinary rows: one pair per C tile).
    if (A->tiles && B->tiles) {
        PEM_TRY(pem_tiled_build_srow(ctx, B));
        PEM_TRY(pem_alloc(ctx, &cp, ntr));
        PEM_TRY(pem_alloc(ctx, &cs, ntr));
        PEM_CK(cudaMemsetAsync(cp, 0, ntr * 8, ctx->stream));
        PEM_CK(cudaMemsetAsync(cs, 0, ntr * 8, ctx->stream));
        k_tile_prodcost<<<pem_div_up(A->tiles, 256), 256, 0, ctx->stream>>>(A->col_occ, A->tile_row_idx, A->tile_col_idx, A->tiles,
                                                                          B->tile_row_ptr, B->srow_ptr, cp, cs);
        PEM_LAUNCHED();
        PEM_CK(cudaMemcpyAsync(hp.data(), cp, ntr * 8, cudaMemcpyDeviceToHost, ctx->stream));
        PEM_CK(cudaMemcpyAsync(hs.data(), cs, ntr * 8, cudaMemcpyDeviceToHost, ctx->stream));
        PEM_CK(cudaStreamSynchronize(ctx->stream));
        pem_free(ctx, cp);
        pem_free(ctx, cs);
    }
    PEM_CK(cudaStreamSynchronize(ctx->stream));
    pem_free(ctx, trf);
    unsigned long long total = 0;
    for (size_t r = 0; r < ntr; ++r) {
        h[r] += 16ull * std::min(hp[r], hs[r]) + 1;  // +1: empty rows still cost a little and keep panels contiguous
        total += h[r];
    }
    bounds[0] = 0;
    unsigned long long run = 0;
    int part = 1;
    for (int r = 0; r < A->tile_rows && part < nparts; ++r) {
        run += h[(size_t)r];
        // close panel `part` once it has reached its share of the prefix
        while (part < nparts && run * (unsigned long long)nparts >= total * (unsigned long long)part) bounds[part++] = r + 1;
    }
    while (part <= nparts) bounds[part++] = A->tile_rows;
    return PEM_OK;
}

}  // extern "C"
