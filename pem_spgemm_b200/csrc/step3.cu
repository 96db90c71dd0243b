// Step 3, numeric: C's values.  Replaces pem_spgemm_step3_accumulate (/root/reference/spgemm.cu:593-661).
//
// Every C nonzero has exactly one owner thread, which adds its products in ascending (pair, k) order
// with one fma each, starting from +0.0: the reference's order (:648-656) and the host oracle's, so the
// value bits agree; C is written exactly once (the reference read-modify-writes global C per product and
// never zeroes it) and no floating-point atomic exists.
//
// Default kernels (chosen per product, pem_step3_numeric): k_step3_windows for dense-tile products (stencil / FEM:
// a block per 128-pair window, the pairs' records staged in shared memory) and k_step3_entries for hypersparse
// tiles (one thread per C nonzero over the flat nonzero index space: every lane of every warp owns one nonzero
// whatever the tile sizes are).  Both defer the fma by one product, so that a warp is not parked behind every
// pair of value gathers (profiles/r02_step3_windows.md).
//
// Selectable (PEM_OPT_OWNER = 3) and bit-identical: k_step3_classes.  A warp takes 32 consecutive C' tiles;
// their offsets are read coalesced and every tile is handled by the mapping its size calls for:
//   small tile   (<= S nonzeros and a short pair list): ONE THREAD per tile, which walks the tile's
//                Ctiles_rowColIdx bytes; single-pair tiles need no hit words.
//   staged tile  (more nonzeros, <= 32 pairs; stencil / FEM products: ~76 nonzeros and 4-5 pairs):
//                ONE WARP per tile.  The A row records and B column records of all its pairs (64 + 64
//                bytes per pair, one coalesced load per pair) and the value offsets are staged in shared
//                memory; lanes own nonzeros (32 per pass) and read records from shared memory only.
//   hub tile     (long pair list): one warp per tile, lanes own nonzeros and find the pairs that feed
//                them by ANDing two words of the bit-transposed hit blocks step 2 left behind.
// Measured on B200 (config 4: 12.1 ms against 12.7 ms; config 2: 5.1 ms against 1.3 ms, hub tiles serialise
// on single warps), so it stays an option.  Also selectable: the row-owner kernel (sixteen lanes per tile).
#include <algorithm>
#include <climits>

#include "engine.cuh"

namespace {

// all products of one (A tile row record, B tile column record) combination, ascending k.
// Records (pem_tiled_build_views): A row record = row mask | first-value offset << 16 (offset < 256: bits 16-23),
// B column record = column mask | first-value offset << 24.  The two offsets sit in different bytes, so the AND of
// two records IS the intersection of the masks: one LOP3 yields the common k's and the "any?" predicate.
// (ao, bo = index of the tiles' first values)
template <class T>
__device__ __forceinline__ T pair_products(unsigned ar, unsigned bc, unsigned ao, unsigned bo,
                                           const T* __restrict__ A_vals, const T* __restrict__ B_vals_t, T acc)
{
    unsigned m = ar & bc;
    if (m) {
        const unsigned ia = ao + (ar >> 16);             // row r of the A tile
        const unsigned ib = bo + (bc >> 24);             // column c of the B tile (values column-major)
        do {
            const unsigned t = m - 1u;
            const unsigned lt = ~m & t;                  // the bits below the lowest common k (lt < 2^16: the offset bits drop out of the ranks)
            m &= t;
            acc = fma(A_vals[ia + __popc(ar & lt)], B_vals_t[ib + __popc(bc & lt)], acc);
        } while (m);
    }
    return acc;
}

__device__ __forceinline__ unsigned lds_u32(uint32_t addr)
{
    unsigned v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ uint2 lds_v2(uint32_t addr)
{
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr) : "memory");
    return v;
}

// Window kernel: the same products with the fma DEFERRED by one product.  A warp issues in order, so an fma placed
// right behind its two value gathers parks the warp for a full memory latency per product (46 % of the kernel's
// stall samples sat there).  Here the gathers of product n are issued, and consumed only when product n + 1 has
// computed its addresses (possibly several pairs later): (pa, pb) hold the operands still in flight.  Same fma
// chain in the same order, preceded by fma(0, 0, +0) = +0, so the value bits do not change.
template <class T>
__device__ __forceinline__ void pair_products_deferred(unsigned m, unsigned ar, unsigned bc, unsigned ao, unsigned bo,
                                                       const T* __restrict__ A_vals, const T* __restrict__ B_vals_t,
                                                       T& acc, T& pa, T& pb)
{
    const unsigned ia = ao + (ar >> 16), ib = bo + (bc >> 24);
    do {
        const unsigned t = m - 1u;
        const unsigned lt = ~m & t;
        m &= t;
        const T* __restrict__ xa = A_vals + (ia + __popc(ar & lt));
        const T* __restrict__ xb = B_vals_t + (ib + __popc(bc & lt));
        acc = fma(pa, pb, acc);
        pa = __ldg(xa);
        pb = __ldg(xb);
    } while (m);
}

// one C nonzero (r, c) of a tile with pairs [ps, pe): the candidate pairs come from the hit blocks
// (word 16+r of 32-pair block b has bit i set iff pair 32b+i touches C row r; word c likewise for columns)
template <class T, bool HITS = true, bool DEFER = true>     // DEFER: fma one product behind its gathers (off in the window kernel's rare path: registers)
__device__ __forceinline__ T entry_by_hits(unsigned r, unsigned c, int64_t ps, int64_t pe,
                                           const int2* __restrict__ pairs, const uint32_t* __restrict__ hit_t,
                                           const uint32_t* __restrict__ A_off, const T* __restrict__ A_vals,
                                           const uint32_t* __restrict__ A_row_rec,
                                           const uint32_t* __restrict__ B_off, const T* __restrict__ B_vals_t,
                                           const uint32_t* __restrict__ B_col_rec)
{
    T acc = 0, pa = 0, pb = 0;                      // (pa, pb): operands of the product whose gathers are in flight
    for (int64_t base = ps & ~(int64_t)31; base < pe; base += 32) {
        unsigned w = HITS ? hit_t[base + 16 + r] & hit_t[base + c] : 0xFFFFFFFFu;    // no hit blocks (dense-tile mode of step 2): every pair is a candidate
        if (base < ps) w &= 0xFFFFFFFFu << (unsigned)(ps - base);
        if (base + 32 > pe) w &= 0xFFFFFFFFu >> (unsigned)(base + 32 - pe);
        while (w) {
            const int64_t i = base + (__ffs(w) - 1);
            w &= w - 1;
            const int2 ab = pairs[i];
            const unsigned ar = A_row_rec[(unsigned)ab.x * 16u + r];
            const unsigned bc = B_col_rec[(unsigned)ab.y * 16u + c];
            const unsigned ao = A_off[ab.x], bo = B_off[ab.y];      // issued with the records, not after the mask test
            if (DEFER) {
                const unsigned m = ar & bc;
                if (m) pair_products_deferred<T>(m, ar, bc, ao, bo, A_vals, B_vals_t, acc, pa, pb);
            } else {
                acc = pair_products(ar, bc, ao, bo, A_vals, B_vals_t, acc);
            }
        }
    }
    return DEFER ? fma(pa, pb, acc) : acc;
}

constexpr int S3C_THREADS = 128;      // four warps, 32 tiles each
constexpr int S3C_WARPS = S3C_THREADS / 32;
constexpr int S3C_NP = 32;            // pairs whose records are staged at once

struct S3CWarp {
    uint32_t rec[S3C_NP][32];         // pair j: A row records at [j][0..15], B column records at [j][16..31]
    uint2 off[S3C_NP];                // pair j: first value of the A tile, of the B tile
};

template <int MINB>
__global__ void __launch_bounds__(S3C_THREADS, MINB)
k_step3_classes(int64_t n_tiles, int small_e, int small_np,
                const int64_t* __restrict__ c_tile_nnz_ptr, const uint4* __restrict__ Cmasks128,
                const uint8_t* __restrict__ c_row_col_idx,
                const int64_t* __restrict__ pair_ptr, const int2* __restrict__ pairs, const uint32_t* __restrict__ hit_t,
                const uint32_t* __restrict__ A_off, const double* __restrict__ A_vals, const uint32_t* __restrict__ A_row_rec,
                const uint32_t* __restrict__ B_off, const double* __restrict__ B_vals_t, const uint32_t* __restrict__ B_col_rec,
                double* __restrict__ C_vals)
{
    __shared__ S3CWarp s_all[S3C_WARPS];
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    S3CWarp& s = s_all[warp];
    const int64_t tbase = ((int64_t)blockIdx.x * S3C_WARPS + warp) * 32;
    if (tbase >= n_tiles) return;                   // whole warps leave together
    const int64_t t = tbase + lane;
    const bool valid = t < n_tiles;
    const int64_t nz0 = valid ? c_tile_nnz_ptr[t] : 0, nz1 = valid ? c_tile_nnz_ptr[t + 1] : 0;
    const int64_t ps = valid ? pair_ptr[t] : 0, pe = valid ? pair_ptr[t + 1] : 0;
    const int E = (int)(nz1 - nz0);
    const int64_t np = pe - ps;
    const bool small = E > 0 && E <= small_e && np <= (int64_t)small_np;
    const bool big = E > 0 && !small;

    // ---- small tiles: one thread per tile ------------------------------------------------------------
    if (small) {
        double* __restrict__ out = C_vals + nz0;
        const uint8_t* __restrict__ rcs = c_row_col_idx + nz0;
        if (np == 1) {
            const int2 ab = pairs[ps];
            const uint32_t* __restrict__ arec = A_row_rec + (size_t)(unsigned)ab.x * 16u;
            const uint32_t* __restrict__ brec = B_col_rec + (size_t)(unsigned)ab.y * 16u;
            const unsigned ao = A_off[ab.x], bo = B_off[ab.y];
            for (int e = 0; e < E; ++e) {
                const unsigned rcb = rcs[e];
                out[e] = pair_products<double>(arec[rcb >> 4], brec[rcb & 15u], ao, bo, A_vals, B_vals_t, 0.0);
            }
        } else {
            for (int e = 0; e < E; ++e) {
                const unsigned rcb = rcs[e];
                out[e] = entry_by_hits<double>(rcb >> 4, rcb & 15u, ps, pe, pairs, hit_t,
                                               A_off, A_vals, A_row_rec, B_off, B_vals_t, B_col_rec);
            }
        }
    }

    // ---- the other tiles of these 32: one warp per tile, one after the other --------------------------
    unsigned todo = __ballot_sync(FULL, big);
    while (todo) {
        const int src = __ffs(todo) - 1;
        todo &= todo - 1;
        const int Et = __shfl_sync(FULL, E, src);
        const int64_t nzt = __shfl_sync(FULL, nz0, src);
        const int64_t pst = __shfl_sync(FULL, ps, src);
        const int64_t npt = __shfl_sync(FULL, np, src);
        double* __restrict__ out = C_vals + nzt;
        const uint8_t* __restrict__ rcs = c_row_col_idx + nzt;
        if (npt <= S3C_NP) {
            // stage the records and value offsets of every pair
            const int npi = (int)npt;
            int2 ab = make_int2(0, 0);
            __syncwarp();                           // the previous tile's readers are done
            if (lane < npi) {
                ab = pairs[pst + lane];
                s.off[lane] = make_uint2(A_off[ab.x], B_off[ab.y]);
            }
            const uint32_t* __restrict__ recs = lane < 16 ? A_row_rec : B_col_rec;
#pragma unroll 4
            for (int j = 0; j < npi; ++j) {
                const unsigned a = (unsigned)__shfl_sync(FULL, ab.x, j), b = (unsigned)__shfl_sync(FULL, ab.y, j);
                s.rec[j][lane] = recs[(lane < 16 ? a : b) * 16u + (unsigned)(lane & 15)];
            }
            __syncwarp();
            for (int e0 = 0; e0 < Et; e0 += 32) {
                const int e = e0 + lane;
                const bool active = e < Et;
                const unsigned rcb = active ? rcs[e] : 0u;
                const uint32_t* sa = &s.rec[0][rcb >> 4];
                const uint32_t* sb = &s.rec[0][16u + (rcb & 15u)];
                const uint2* so = &s.off[0];
                double acc = 0.0;
                for (int j = 0; j < npi; ++j, sa += 32, sb += 32, ++so) {
                    const unsigned ar = *sa, bc = *sb;
                    unsigned m = active ? (ar & bc) : 0u;
                    if (m) {
                        const uint2 o = *so;
                        const unsigned ia = o.x + (ar >> 16), ib = o.y + (bc >> 24);     // 32-bit value indices
                        do {
                            const unsigned low = m & (0u - m);
                            m ^= low;
                            const unsigned lt = low - 1u;
                            acc = fma(A_vals[ia + __popc(ar & lt)], B_vals_t[ib + __popc(bc & lt)], acc);
                        } while (m);
                    }
                }
                if (active) out[e] = acc;
            }
        } else {
            for (int e0 = 0; e0 < Et; e0 += 32) {
                const int e = e0 + lane;
                if (e < Et) {
                    const unsigned rcb = rcs[e];
                    out[e] = entry_by_hits<double>(rcb >> 4, rcb & 15u, pst, pst + npt, pairs, hit_t,
                                                   A_off, A_vals, A_row_rec, B_off, B_vals_t, B_col_rec);
                }
            }
        }
    }
}

// =========================================================================================
// PEM_OPT_OWNER = 2: one thread per C nonzero over the flat nonzero index space (round 1's default).
// The block covers S3E_ENTRIES consecutive nonzeros; the offsets of the tiles it overlaps are staged in
// shared memory and each thread finds its tile by binary search there; its (r, c) is Ctiles_rowColIdx[n].
// =========================================================================================
constexpr int S3E_ENTRIES = 128;
constexpr int S3E_TMAX = 512;

// first tile of every entry-owner block (a tile of up to 256 nonzeros can cover two block boundaries)
__global__ void __launch_bounds__(256)
k_block_tiles(int64_t n_tiles, const int64_t* __restrict__ c_tile_nnz_ptr, int32_t* __restrict__ blk_tile)
{
    int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_tiles) return;
    const int64_t off = c_tile_nnz_ptr[t], end = c_tile_nnz_ptr[t + 1];
    if (end > off) {
        for (int64_t bnd = (off + S3E_ENTRIES - 1) / S3E_ENTRIES * S3E_ENTRIES; bnd < end; bnd += S3E_ENTRIES)
            blk_tile[bnd / S3E_ENTRIES] = (int32_t)t;
    }
}

template <class T>          // value type: double (the reference's ValueType, spgemm.cu:728) or float
__global__ void __launch_bounds__(S3E_ENTRIES, 16)
k_step3_entries(int64_t nnz, int64_t n_tiles, const int32_t* __restrict__ blk_tile,
                const int64_t* __restrict__ c_tile_nnz_ptr, const uint8_t* __restrict__ c_row_col_idx,
                const uint32_t* __restrict__ Cmasks32,
                const int64_t* __restrict__ pair_ptr, const int2* __restrict__ pairs,
                const uint32_t* __restrict__ hit_t,
                const uint32_t* __restrict__ A_off, const T* __restrict__ A_vals,
                const uint32_t* __restrict__ A_row_rec,
                const uint32_t* __restrict__ B_off, const T* __restrict__ B_vals_t,
                const uint32_t* __restrict__ B_col_rec, T* __restrict__ C_vals)
{
    constexpr bool RC = false;      // (r, c) from the tile mask; reading Ctiles_rowColIdx instead is 8 % faster here but producing it costs more
    __shared__ int s_off[S3E_TMAX];
    const int tid = threadIdx.x;
    const int64_t n0 = (int64_t)blockIdx.x * S3E_ENTRIES;
    const int64_t t0 = blk_tile[blockIdx.x];
    const int64_t t1 = (n0 + S3E_ENTRIES < nnz) ? (int64_t)blk_tile[blockIdx.x + 1] : n_tiles - 1;
    const int64_t span = t1 - t0 + 1;
    const bool staged = span <= S3E_TMAX;
    if (staged)
        for (int i = tid; i < (int)span; i += S3E_ENTRIES) s_off[i] = (int)(c_tile_nnz_ptr[t0 + i] - n0);
    __syncthreads();
    const int64_t n = n0 + tid;
    if (n >= nnz) return;
    unsigned rcb = 0;
    if (RC) rcb = c_row_col_idx[n];                 // independent of the tile search below: both loads are in flight together
    int64_t t;
    int e;                                          // rank of this nonzero inside its tile
    if (staged) {                                   // last i with s_off[i] <= tid
        int lo = 0, hi = (int)span - 1;
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (s_off[mid] <= tid) lo = mid; else hi = mid - 1;
        }
        t = t0 + lo;
        e = tid - s_off[lo];
    } else {                                        // many empty tiles in range (keep_empty mode)
        int64_t lo = t0, hi = t1;
        while (lo < hi) {
            const int64_t mid = (lo + hi + 1) >> 1;
            if (c_tile_nnz_ptr[mid] <= n) lo = mid; else hi = mid - 1;
        }
        t = lo;
        e = (int)(n - c_tile_nnz_ptr[t]);
    }
    unsigned r, c;
    if (RC) {
        r = rcb >> 4;
        c = rcb & 15u;
    } else {
        // (r, c) = position of the e-th set bit of the tile's 256-bit mask (word w = rows 2w, 2w+1), which
        // is what Ctiles_rowColIdx[n] holds (spgemm.cu:552-591), without materialising that array
        const uint4* m4 = reinterpret_cast<const uint4*>(Cmasks32 + (size_t)t * 8);
        const uint4 x = m4[0], y = m4[1];
        const unsigned w[8] = {x.x, x.y, x.z, x.w, y.x, y.y, y.z, y.w};
        unsigned sel = 0, wi = 0;
        int rem = e;
        bool done = false;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int pc = __popc(w[i]);
            const bool here = !done && rem < pc;
            sel = here ? w[i] : sel;
            wi = here ? (unsigned)i : wi;
            done = done || here;
            rem -= done ? 0 : pc;
        }
        unsigned b = 0;                             // position of the rem-th set bit of sel: 5 halving steps
#pragma unroll
        for (int width = 16; width > 0; width >>= 1) {
            const int pc = __popc(sel & (((1u << width) - 1u) << b));
            const bool up = rem >= pc;
            rem -= up ? pc : 0;
            b += up ? (unsigned)width : 0u;
        }
        r = 2u * wi + (b >> 4);
        c = b & 15u;
    }
    C_vals[n] = entry_by_hits<T>(r, c, pair_ptr[t], pair_ptr[t + 1], pairs, hit_t,
                                 A_off, A_vals, A_row_rec, B_off, B_vals_t, B_col_rec);
}

// =========================================================================================
// PEM_OPT_OWNER = 4: WINDOW kernel.  A block takes one window of the pair list: the C' tiles whose first
// pair lies in [w * NP, (w + 1) * NP) (at most NP tiles, found through k_window_tiles' table).  The block
//   1. stages, for every pair of the window, A's sixteen row records and B's sixteen column records
//      (128 bytes per pair, eight lanes per pair, 128-bit asynchronous copies) and the two value offsets in
//      shared memory, next to the tiles' masks, pair ranges and nonzero offsets;
//   2. decodes the window's nonzeros cooperatively while those copies are in flight: one lane per 32-bit
//      mask word (two tile rows), the word's rank by an 8-lane scan, one 16-bit code
//      (tile << 8 | r << 4 | c) per nonzero;
//   3. lets every thread own nonzeros (consecutive threads = consecutive nonzeros, so C is written
//      coalesced): the pair loop and both record reads run out of shared memory, only the two value
//      gathers per product touch global memory.
// No per-thread tile search, no rank select, no hit words; the dependent chain of the entry-owner kernel
// (tile offset -> mask -> hit words -> pair -> records -> values, paid per nonzero with a global-memory
// latency each) becomes window -> pairs -> records, taken once per window with all loads of a stage in
// flight together, then values.  The pair loop runs on three shared-memory addresses and tests a pair with one
// LOP3 (record offsets in disjoint bytes); the fma runs one product behind its gathers.  The window's last tile
// may own more pairs than are staged (hub tiles of power-law inputs, wide dense bands): it is computed through the
// hit blocks like the entry-owner kernel does, or, when step 2 ran in dense-tile mode and left none (HITS = false),
// by testing every pair of the tile.
// Measured and rejected (profiles/r02_step3_windows.md): the tiles' VALUES staged in shared memory as well
// (8-byte cp.async, packed per warp: the ~65 instructions per pair of the copy loop cost more than the
// load stalls they remove, 19.1 ms against 11.2 ms on config 4), 1-D bulk copies (cp.async.bulk) for the
// per-pair payloads (a warp issues them one lane at a time, ~36 ns per copy, tools/ubench/bulk_rate.cu), value base
// addresses pinned in 64-bit registers, streaming hints, the unstaged path out of line.
// =========================================================================================
constexpr int S3W_THREADS = 256;

// win_tile[w] = first tile whose pair list starts at or after pair w * np (w = 0 .. n_windows)
__global__ void __launch_bounds__(256)
k_window_tiles(int64_t n_tiles, int64_t n_windows, int np, const int64_t* __restrict__ pair_ptr, int32_t* __restrict__ win_tile)
{
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t > n_tiles) return;
    const int64_t lo = t == 0 ? 0 : pair_ptr[t - 1] / np + 1;
    const int64_t hi = min(pair_ptr[t] / np, n_windows);
    for (int64_t w = lo; w <= hi; ++w) win_tile[w] = (int32_t)t;
    if (t == n_tiles) win_tile[n_windows] = (int32_t)n_tiles;
}

__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_addr(smem_dst)), "l"(gmem_src) : "memory");
}

// shared-memory layout of the window kernel
template <int NP, int SCAP, int ECAP>
struct S3WLayout {
    static constexpr int REC = 0;
    static constexpr int VOFF = REC + SCAP * 128;
    static constexpr int MASK = VOFF + SCAP * 8;
    static constexpr int PP = MASK + NP * 32;
    static constexpr int NZ = PP + (NP + 4) * 4;
    static constexpr int CODE = NZ + (NP + 4) * 4;
    static constexpr int BYTES = CODE + ECAP * 2;
};

template <class T, int NP, int SCAP, int ECAP, int MINB, bool HITS>   // window pairs, staged pairs (multiple of 16), nonzeros decoded per pass, hit blocks present
__global__ void __launch_bounds__(S3W_THREADS, MINB)
k_step3_windows(const int32_t* __restrict__ win_tile, const int64_t* __restrict__ c_tile_nnz_ptr,
                const uint4* __restrict__ Cmasks128, const int64_t* __restrict__ pair_ptr,
                const int2* __restrict__ pairs, const uint32_t* __restrict__ hit_t,
                const uint32_t* __restrict__ A_off, const T* __restrict__ A_vals, const uint4* __restrict__ A_row_rec4,
                const uint32_t* __restrict__ B_off, const T* __restrict__ B_vals_t, const uint4* __restrict__ B_col_rec4,
                T* __restrict__ C_vals, unsigned vsz)
{
    static_assert(SCAP % 16 == 0 && SCAP >= NP && (SCAP + 31) / 32 <= S3W_THREADS / 32 && NP <= 128, "window shape");
    using L = S3WLayout<NP, SCAP, ECAP>;
    static_assert(L::REC == 0, "the pair loop derives the staged pair index from the record's byte offset");
    extern __shared__ __align__(128) unsigned char s_raw[];
    uint32_t* s_rec = reinterpret_cast<uint32_t*>(s_raw + L::REC);     // pair j: A row records [32j .. 32j+15], B column records [32j+16 .. 32j+31]
    uint2* s_voff = reinterpret_cast<uint2*>(s_raw + L::VOFF);         // pair j: first value of the A tile, of the B tile
    uint32_t* s_mask = reinterpret_cast<uint32_t*>(s_raw + L::MASK);
    int* s_pp = reinterpret_cast<int*>(s_raw + L::PP);                 // pair ranges, relative to the window's first pair
    int* s_nz = reinterpret_cast<int*>(s_raw + L::NZ);                 // nonzero offsets, relative to the window's first nonzero
    uint16_t* s_code = reinterpret_cast<uint16_t*>(s_raw + L::CODE);
    const unsigned FULL = 0xffffffffu;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t sbase = smem_addr(s_raw);                            // 128-byte aligned
    const int64_t ta = win_tile[blockIdx.x], tb = win_tile[blockIdx.x + 1];
    const int nt = (int)(tb - ta);
    if (nt <= 0) return;                                        // a hub tile spans this whole window
    const int64_t P0 = pair_ptr[ta], N0 = c_tile_nnz_ptr[ta];
    const int64_t p_last = pair_ptr[tb] - P0, p_prev = pair_ptr[tb - 1] - P0;
    const int ns = p_last <= SCAP ? (int)p_last : (int)p_prev;  // staged pairs (p_prev < NP)
    // ---- 1. asynchronous copies: records of the window's pairs; their value offsets ---------------------
    if (warp * 32 < ns) {
        const int j0 = warp * 32, jm = j0 + lane;
        int2 ab = make_int2(0, 0);
        if (jm < ns) ab = pairs[P0 + jm];
        const int part = lane & 7;
#pragma unroll
        for (int q = 0; q < 8; ++q) {                           // four pairs per warp-wide 128-bit copy
            const int jl = q * 4 + (lane >> 3);
            const unsigned ax = (unsigned)__shfl_sync(FULL, ab.x, jl), by = (unsigned)__shfl_sync(FULL, ab.y, jl);
            if (j0 + jl < ns)
                cp_async16(reinterpret_cast<uint4*>(s_rec) + (j0 + jl) * 8 + part,
                           part < 4 ? A_row_rec4 + (size_t)ax * 4 + part : B_col_rec4 + (size_t)by * 4 + (part - 4));
        }
        if (jm < ns) s_voff[jm] = make_uint2(A_off[ab.x], B_off[ab.y]);
    }
    for (int x = tid; x <= nt; x += S3W_THREADS) {
        s_pp[x] = (int)min(pair_ptr[ta + x] - P0, (int64_t)0x3fffffff);
        s_nz[x] = (int)(c_tile_nnz_ptr[ta + x] - N0);
    }
    for (int x = tid; x < nt * 2; x += S3W_THREADS) reinterpret_cast<uint4*>(s_mask)[x] = Cmasks128[ta * 2 + x];
    __syncthreads();
    const int ne = s_nz[nt];
    for (int e0 = 0; e0 < ne; e0 += ECAP) {
        // ---- 2. decode: lane = one mask word (rows 2w, 2w+1) of one tile ---------------------------------
        for (int it0 = warp * 32; it0 < nt * 8; it0 += S3W_THREADS) {
            const int it = it0 + lane;
            unsigned word = it < nt * 8 ? s_mask[it] : 0u;
            const int pc = __popc(word);
            int incl = pc;
#pragma unroll
            for (int o = 1; o < 8; o <<= 1) {
                const int v = __shfl_up_sync(FULL, incl, o, 8);
                if ((lane & 7) >= o) incl += v;
            }
            if (word) {
                int rank = s_nz[it >> 3] + (incl - pc) - e0;
                const unsigned base = (unsigned)(it >> 3) << 8 | (unsigned)(it & 7) << 5;
                if (ne <= ECAP) {                       // one pass (the usual case): every rank is in range
                    uint16_t* dst = s_code + rank;
                    do {
                        const unsigned b = __ffs(word) - 1;
                        word &= word - 1;
                        *dst++ = (uint16_t)(base + b);
                    } while (word);
                } else {
                    do {
                        const unsigned b = __ffs(word) - 1;
                        word &= word - 1;
                        if ((unsigned)rank < (unsigned)ECAP) s_code[rank] = (uint16_t)(base + b);
                        ++rank;
                    } while (word);
                }
            }
        }
        if (e0 == 0) asm volatile("cp.async.wait_all;" ::: "memory");
        __syncthreads();
        // ---- 3. one thread per nonzero ------------------------------------------------------------------
        const int e1 = min(ne, e0 + ECAP);
        for (int i = e0 + tid; i < e1; i += S3W_THREADS) {
            const unsigned code = s_code[i - e0];
            const unsigned tl = code >> 8;
            const int js = s_pp[tl], je = s_pp[tl + 1];
            T acc = 0;
            if (je <= ns) {
                // the pair loop runs on three shared-memory ADDRESSES (A row record, B column record, value offsets of the
                // current pair) and one compare; a hit is one LOP3 (the records' offsets sit in disjoint bytes)
                uint32_t ra = sbase + (unsigned)js * 128u + ((code >> 2) & 0x3Cu);
                uint32_t rb = sbase + (unsigned)js * 128u + 64u + ((code & 15u) << 2);
                uint32_t va = sbase + L::VOFF + (unsigned)js * 8u;
                const uint32_t ra_end = ra + (unsigned)(je - js) * 128u;
                T pa = 0, pb = 0;                       // operands of the product whose gathers are in flight
                while (ra != ra_end) {
                    const unsigned ar = lds_u32(ra), bc = lds_u32(rb);
                    const unsigned m = ar & bc;
                    if (m) {
                        const uint2 o = lds_v2(va);
                        pair_products_deferred<T>(m, ar, bc, o.x, o.y, A_vals, B_vals_t, acc, pa, pb);
                    }
                    ra += 128u;
                    rb += 128u;
                    va += 8u;
                }
                acc = fma(pa, pb, acc);
            } else {
                // the window's last tile owns more pairs than are staged (hub tiles of power-law inputs, wide dense bands): through
                // the hit blocks like the entry-owner kernel, or over every pair of the tile when step 2 produced no hit blocks
                acc = entry_by_hits<T, HITS, false>((code >> 4) & 15u, code & 15u, pair_ptr[ta + tl], pair_ptr[ta + tl + 1], pairs, hit_t,
                                             A_off, A_vals, reinterpret_cast<const uint32_t*>(A_row_rec4),
                                             B_off, B_vals_t, reinterpret_cast<const uint32_t*>(B_col_rec4));
            }
            C_vals[N0 + i] = acc;
        }
        if (e0 + ECAP < ne) __syncthreads();
    }
}

// one window-kernel configuration: table kernel + numeric kernel
template <class T, int NP, int SCAP, int ECAP, int MINB, bool HITS>
static int launch_windows(pem_ctx* ctx, const pem_tiled* A, const pem_tiled* B, pem_result* C)
{
    const int64_t n_windows = (C->pairs + NP - 1) / NP;
    if (n_windows > 0x7fffffffLL) return ctx->fail(PEM_ERR_LIMIT, "more than 2^37 tile pairs");
    int32_t* win_tile = nullptr;
    pem_guard g(ctx, win_tile);
    PEM_TRY(pem_alloc(ctx, &win_tile, (size_t)n_windows + 1));
    k_window_tiles<<<pem_div_up(C->tiles + 1, 256), 256, 0, ctx->stream>>>(C->tiles, n_windows, NP, C->pair_ptr, win_tile);
    PEM_LAUNCHED();
    auto kern = k_step3_windows<T, NP, SCAP, ECAP, MINB, HITS>;
    constexpr int smem = S3WLayout<NP, SCAP, ECAP>::BYTES;
    // window shapes above 48 KB of dynamic shared memory opt in (per launch: the attribute belongs to the device the
    // context runs on, and a process may hold one context per GPU; the shipped 26 KB shape compiles this away)
    if constexpr (smem > 48 * 1024) PEM_CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    KT_BEGIN(KT_NUMERIC);
    kern<<<(unsigned)n_windows, S3W_THREADS, smem, ctx->stream>>>(
        win_tile, C->tile_nnz_ptr, reinterpret_cast<const uint4*>(C->masks), C->pair_ptr, C->pair_list, C->pair_hit,
        A->tile_nnz_ptr, reinterpret_cast<const T*>(A->vals), reinterpret_cast<const uint4*>(A->row_rec),
        B->tile_nnz_ptr, reinterpret_cast<const T*>(B->vals_t), reinterpret_cast<const uint4*>(B->col_rec),
        reinterpret_cast<T*>(C->vals), (unsigned)sizeof(T));
    KT_END(KT_NUMERIC);
    PEM_LAUNCHED();
    pem_free(ctx, win_tile);
    return PEM_OK;
}

// =========================================================================================
// PEM_OPT_OWNER = 1: SIXTEEN LANES PER C' TILE, lane = row r of the tile (two tiles per warp), paired
// with k_step2_masks in step 2.  Lane r accumulates its C row in FOUR REGISTERS: the nonzeros of the row
// are numbered by rank inside Cmask[r] and handled four ranks per pass.  An independent formulation of
// steps 2 and 3 (no pair kernel, no hit blocks, no records) kept as a cross-check of the default path.
// =========================================================================================
constexpr int S3_THREADS = 256;
constexpr int S3_NACC = 4;

__global__ void __launch_bounds__(S3_THREADS)
k_step3_numeric(int64_t n_tiles, const int64_t* __restrict__ pair_ptr, const int2* __restrict__ pairs,
                const uint16_t* __restrict__ Cmasks, const int64_t* __restrict__ c_tile_nnz_ptr,
                const uint32_t* __restrict__ A_off, const double* __restrict__ A_vals,
                const uint16_t* __restrict__ A_masks, const uint8_t* __restrict__ A_rowptr,
                const uint32_t* __restrict__ B_off, const double* __restrict__ B_vals,
                const uint16_t* __restrict__ B_masks, const uint8_t* __restrict__ B_rowptr,
                double* __restrict__ C_vals)
{
    const int tid = threadIdx.x;
    const int64_t t = ((int64_t)blockIdx.x * S3_THREADS + tid) >> 4;
    const unsigned r = tid & 15u;
    if (t >= n_tiles) return;                       // whole 16-lane groups leave together
    const unsigned grp = 0xFFFFu << (tid & 16);
    const unsigned cm = Cmasks[t * 16 + r];
    // offset of row r inside the tile: exclusive scan of the row popcounts over the 16 lanes
    const int pc = __popc(cm);
    int incl = pc;
#pragma unroll
    for (int o = 1; o < 16; o <<= 1) {
        const int v = __shfl_up_sync(grp, incl, o, 16);
        if ((int)r >= o) incl += v;
    }
    if (cm == 0) return;                            // nothing lands in this row
    const int64_t ps = pair_ptr[t];
    const unsigned np = (unsigned)(pair_ptr[t + 1] - ps);
    const int2* __restrict__ pl = pairs + ps;
    double* __restrict__ out = C_vals + c_tile_nnz_ptr[t] + (incl - pc);
    unsigned rest = cm;                             // columns not yet produced
    for (int lo = 0; lo < pc; lo += S3_NACC) {
        // the (up to) four lowest remaining columns form this pass
        unsigned pm = 0;
#pragma unroll
        for (int j = 0; j < S3_NACC; ++j) {
            const unsigned low = rest & (0u - rest);
            pm |= low;
            rest ^= low;
        }
        double acc0 = 0.0, acc1 = 0.0, acc2 = 0.0, acc3 = 0.0;
        int2 ab_n = pl[0];
        unsigned am_n = A_masks[(unsigned)ab_n.x * 16u + r];
        for (unsigned i = 0; i < np; ++i) {
            const int2 ab = ab_n;
            unsigned am = am_n;
            if (i + 1 < np) {                       // prefetch the next pair
                ab_n = pl[i + 1];
                am_n = A_masks[(unsigned)ab_n.x * 16u + r];
            }
            if (am) {
                const unsigned ib = (unsigned)ab.y * 16u;
                const double* __restrict__ ap = A_vals + (A_off[ab.x] + A_rowptr[(unsigned)ab.x * 16u + r]);
                const double* __restrict__ bbase = B_vals + B_off[ab.y];
                do {
                    const unsigned k = __ffs(am) - 1;
                    am &= am - 1;
                    const unsigned bm = B_masks[ib + k];
                    unsigned hit = bm & pm;
                    if (hit) {
                        const double a = *ap;
                        const double* __restrict__ bp = bbase + B_rowptr[ib + k];
                        do {
                            const unsigned low = hit & (0u - hit);
                            hit ^= low;
                            const double b = bp[__popc(bm & (low - 1u))];
                            const int idx = __popc(pm & (low - 1u));
                            const double v0 = fma(a, b, acc0), v1 = fma(a, b, acc1), v2 = fma(a, b, acc2), v3 = fma(a, b, acc3);
                            acc0 = idx == 0 ? v0 : acc0;
                            acc1 = idx == 1 ? v1 : acc1;
                            acc2 = idx == 2 ? v2 : acc2;
                            acc3 = idx == 3 ? v3 : acc3;
                        } while (hit);
                    }
                    ++ap;
                } while (am);
            }
        }
        const int cnt = min(S3_NACC, pc - lo);
        out[0] = acc0;
        if (cnt > 1) out[1] = acc1;
        if (cnt > 2) out[2] = acc2;
        if (cnt > 3) out[3] = acc3;
        out += S3_NACC;
    }
}

}  // namespace

extern "C" int pem_step3_numeric(pem_ctx* ctx, const pem_tiled* A, const pem_tiled* B, pem_result* C)
{
    PEM_RANGE("pem_step3_numeric");
    if (!ctx || !A || !B || !C) return PEM_ERR_ARG;
    if (C->stage != 2) return ctx->fail(PEM_ERR_ARG, "step 3 needs a result fresh from step 2");
    PEM_CK(cudaSetDevice(ctx->device));
    PEM_TRY(pem_tiled_wait_vals(ctx, A));        // freshly converted operands: the values may still be on their way
    PEM_TRY(pem_tiled_wait_vals(ctx, B));
    if (C->dtype == PEM_F32 && (!C->s2_pairs || !C->s3_entries))
        return ctx->fail(PEM_ERR_ARG, "fp32 products run the default kernels only (PEM_OPT_OWNER 0 / 2 / 4)");
    const bool by_records = C->s2_pairs;                    // step 2 ran the pair kernel
    // dense-tile mode of step 2 (no hit words): only the window kernel can run
    if (by_records && !C->pair_hit && !(C->s3_entries && (ctx->opt_owner == 0 || ctx->opt_owner == 4)))
        return ctx->fail(PEM_ERR_ARG, "step 2 ran in dense-tile mode (no hit words): set PEM_OPT_OWNER before step 2, not between steps 2 and 3");
    // the class kernel reads every nonzero's (r, c) from Ctiles_rowColIdx; the entry-owner kernel derives it
    // from the tile mask (measured on config 4: 11.6 ms against 12.7 ms with the bytes, but producing them costs 1.0 ms)
    const bool use_rc = !C->s3_entries;
    // default: the window kernel when C's tiles are dense enough that staging a pair's 128 bytes of records pays
    // (at least four nonzeros per pair: stencil / FEM products), else the entry-owner kernel
    const bool windows = by_records && C->s3_entries &&
                         (ctx->opt_owner == 4 || !C->pair_hit || (ctx->opt_owner == 0 && C->nnz >= 4 * C->pairs));
    const int64_t nblk_e = (C->nnz + S3E_ENTRIES - 1) / S3E_ENTRIES;      // blocks of the entry-owner kernel
    if (by_records && C->s3_entries && !windows && nblk_e > 0x7fffffffLL) return ctx->fail(PEM_ERR_LIMIT, "C has more than 2^39 nonzeros");
    // buffers of an earlier call that failed part-way: a retry must not overwrite live blocks
    pem_free(ctx, C->vals); pem_free(ctx, C->blk_tile);
    PEM_TRY(pem_alloc_bytes(ctx, (void**)&C->vals, std::max<size_t>(1, (size_t)C->nnz * pem_vsize(C->dtype))));
    if (C->nnz > 0 && by_records) {                          // views are cached on the handles after the first product
        PEM_TRY(pem_tiled_build_views(ctx, A, true, false));
        PEM_TRY(pem_tiled_build_views(ctx, B, false, true));
        if (use_rc) PEM_TRY(pem_result_make_rowcolidx(ctx, C));   // Ctiles_rowColIdx: every nonzero's (r, c), one byte (spgemm.cu:552-591)
    }
    if (C->nnz > 0 && by_records && C->s3_entries && !windows) {   // entry-owner needs the first tile of each of its blocks
        PEM_TRY(pem_alloc(ctx, &C->blk_tile, (size_t)nblk_e + 1));
        k_block_tiles<<<pem_div_up(C->tiles, 256), 256, 0, ctx->stream>>>(C->tiles, C->tile_nnz_ptr, C->blk_tile);
        PEM_LAUNCHED();
    }
    C->s3_kernel = windows ? 4 : !by_records ? 1 : C->s3_entries ? 2 : 3;
    ctx->last_step3_kernel = C->s3_kernel;
    PEM_TRY(pem_step3_launch(ctx, A, B, C));
    C->stage = 3;
    return PEM_OK;
}

// The numeric kernel C->s3_kernel on C's existing buffers: C->vals, the views of A and B, and what that kernel reads
// besides (blk_tile for the entry-owner kernel, row_col_idx for the tile-class kernel) are in place.
int pem_step3_launch(pem_ctx* ctx, const pem_tiled* A, const pem_tiled* B, pem_result* C)
{
    const bool windows = C->s3_kernel == 4, by_records = C->s2_pairs;
    const int64_t nblk_e = (C->nnz + S3E_ENTRIES - 1) / S3E_ENTRIES;
    if (C->nnz > 0 && windows) {
        // 128-pair windows, 144 staged pairs, 1024 nonzeros per decode pass: 26 KB of shared memory and 32 registers, so
        // that eight blocks (64 warps) stay resident per SM: the kernel is bound by the latency of its value gathers, and
        // 8 blocks measured 8.9 ms on config 4 against 10.3 ms with 6 (160 staged pairs, 2048 nonzeros per pass)
        if (C->pair_hit)
            PEM_TRY(C->dtype == PEM_F32 ? (launch_windows<float, 128, 144, 1024, 8, true>(ctx, A, B, C))
                                        : (launch_windows<double, 128, 144, 1024, 8, true>(ctx, A, B, C)));
        else
            PEM_TRY(C->dtype == PEM_F32 ? (launch_windows<float, 128, 144, 1024, 8, false>(ctx, A, B, C))
                                        : (launch_windows<double, 128, 144, 1024, 8, false>(ctx, A, B, C)));
        return PEM_OK;
    }
    KT_BEGIN(KT_NUMERIC);
    if (C->nnz > 0 && by_records && C->s3_entries) {
#define S3E_ARGS C->nnz, C->tiles, C->blk_tile, C->tile_nnz_ptr, C->row_col_idx, reinterpret_cast<const uint32_t*>(C->masks), \
            C->pair_ptr, C->pair_list, C->pair_hit, A->tile_nnz_ptr, A->vals, A->row_rec, B->tile_nnz_ptr, B->vals_t, B->col_rec, C->vals
        if (C->dtype == PEM_F32)
            k_step3_entries<float><<<(unsigned)nblk_e, S3E_ENTRIES, 0, ctx->stream>>>(
                C->nnz, C->tiles, C->blk_tile, C->tile_nnz_ptr, C->row_col_idx, reinterpret_cast<const uint32_t*>(C->masks),
                C->pair_ptr, C->pair_list, C->pair_hit, A->tile_nnz_ptr, reinterpret_cast<const float*>(A->vals), A->row_rec,
                B->tile_nnz_ptr, reinterpret_cast<const float*>(B->vals_t), B->col_rec, reinterpret_cast<float*>(C->vals));
        else
            k_step3_entries<double><<<(unsigned)nblk_e, S3E_ENTRIES, 0, ctx->stream>>>(S3E_ARGS);
#undef S3E_ARGS
        PEM_LAUNCHED();
    } else if (C->nnz > 0 && by_records) {
        const int64_t nblk = (C->tiles + S3C_THREADS - 1) / S3C_THREADS;
#define S3C_ARGS C->tiles, ctx->opt_s3_small_e, ctx->opt_s3_small_np, C->tile_nnz_ptr, reinterpret_cast<const uint4*>(C->masks), \
            C->row_col_idx, C->pair_ptr, C->pair_list, C->pair_hit, A->tile_nnz_ptr, A->vals, A->row_rec, \
            B->tile_nnz_ptr, B->vals_t, B->col_rec, C->vals
        k_step3_classes<10><<<(unsigned)nblk, S3C_THREADS, 0, ctx->stream>>>(S3C_ARGS);     // 10 blocks per SM measured best (8: +9 %, 12: +1 %)
#undef S3C_ARGS
        PEM_LAUNCHED();
    } else if (C->tiles > 0) {
        const int64_t nblk = (C->tiles * 16 + S3_THREADS - 1) / S3_THREADS;
        if (nblk > 0x7fffffffLL) return ctx->fail(PEM_ERR_LIMIT, "C has more than 2^35 tiles");
        k_step3_numeric<<<(unsigned)nblk, S3_THREADS, 0, ctx->stream>>>(
            C->tiles, C->pair_ptr, C->pair_list, C->masks, C->tile_nnz_ptr,
            A->tile_nnz_ptr, A->vals, A->masks, A->row_ptr, B->tile_nnz_ptr, B->vals, B->masks, B->row_ptr, C->vals);
        PEM_LAUNCHED();
    }
    KT_END(KT_NUMERIC);
    return PEM_OK;
}
