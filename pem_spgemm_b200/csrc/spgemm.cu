// The three SpGEMM steps on tiled operands (one iteration of /root/reference/spgemm.cu:1133-1357).
//
//   step 1  tile-level symbolic: lives in step1_esc.cu (default) and step1.cu (small operands).
//   step 2  per-tile bitmask symbolic: C tile masks, per-tile nnz, scan (rowColIdx on request only).
//           Replaces pem_spgemm_step2_compute_CMasksAndOffsets (:499-550) and ..._CrowColIdx
//           (:552-591).  Default mapping: one thread per (A tile, B tile) pair (k_step2_pairs).
//   step 3  numeric: lives in step3.cu.
#include <cub/device/device_scan.cuh>
#include <thrust/iterator/counting_iterator.h>
#include <thrust/iterator/transform_iterator.h>

#include <climits>
#include <memory>
#include <unordered_set>
#include <chrono>
#include <algorithm>

#include "engine.cuh"

namespace {

// =========================================================================================
// PEM_OPT_OWNER = 1: SIXTEEN LANES PER C' TILE in steps 2 and 3, lane = row r of the tile (two tiles
// per warp).  The lane owns row r of the C tile, so no two threads ever update the same C entry:
// atomic-free and, because a lane visits its tile's pairs in list order (ascending k across
// tiles) and the set bits of Amask[r] in ascending k inside a tile, every C entry is accumulated
// in exactly the oracle's order.
// =========================================================================================

// step 2, kernel 1:  Cmask[r] = OR over pairs, OR over k in Amask[r], of Bmask[k]
// (the boolean product of the two 16x16 bit matrices, row by row), and the tile's nnz.
__global__ void __launch_bounds__(256)
k_step2_masks(int64_t n_tiles, const int64_t* __restrict__ pair_ptr, const int2* __restrict__ pairs,
              const uint16_t* __restrict__ Amasks, const uint16_t* __restrict__ Bmasks,
              uint16_t* __restrict__ Cmasks, int64_t* __restrict__ c_tile_nnz)
{
    const int64_t gt = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t t = gt >> 4;
    const unsigned r = threadIdx.x & 15u;
    if (t >= n_tiles) return;                       // whole 16-lane groups leave together
    const unsigned grp = 0xFFFFu << (threadIdx.x & 16u);
    const int64_t ps = pair_ptr[t];
    const unsigned np = (unsigned)(pair_ptr[t + 1] - ps);
    const int2* __restrict__ pl = pairs + ps;
    unsigned acc = 0;
    for (unsigned i = 0; i < np; ++i) {
        const int2 ab = pl[i];
        unsigned m = Amasks[(unsigned)ab.x * 16u + r];
        const uint16_t* __restrict__ bm = Bmasks + (size_t)(unsigned)ab.y * 16u;
        while (m) {
            const unsigned k = __ffs(m) - 1;
            m &= m - 1;
            acc |= bm[k];
        }
    }
    Cmasks[t * 16 + r] = (uint16_t)acc;
    int nnz = __popc(acc);
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) nnz += __shfl_xor_sync(grp, nnz, o, 16);
    if (r == 0) c_tile_nnz[t] = nnz;
}

// Ctiles_rowColIdx ((r<<4)|c per nonzero, row-major inside a tile): part of the reference's data
// contract (spgemm.cu:552-591) but read by nothing in this engine, so it is produced on demand
// only (pem_result_get / tests).  One thread per C' tile, bytes assembled eight at a time.
__global__ void __launch_bounds__(128)
k_rowcolidx(int64_t n_tiles, const uint16_t* __restrict__ Cmasks, const int64_t* __restrict__ c_tile_nnz_ptr,
            uint8_t* __restrict__ row_col_idx)
{
    int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_tiles) return;
    const uint4* m4 = reinterpret_cast<const uint4*>(Cmasks + (size_t)t * 16);
    const uint4 x = m4[0], y = m4[1];
    const unsigned w[8] = {x.x, x.y, x.z, x.w, y.x, y.y, y.z, y.w};
    uint8_t* dst = row_col_idx + c_tile_nnz_ptr[t];
    int head = (int)((8 - ((uintptr_t)dst & 7)) & 7);   // single bytes until dst is 8-byte aligned
    unsigned long long buf = 0;
    int nb = 0;
#pragma unroll
    for (int r = 0; r < 16; ++r) {
        unsigned m = (w[r >> 1] >> ((r & 1) * 16)) & 0xFFFFu;
        while (m) {
            const unsigned c = __ffs(m) - 1;
            m &= m - 1;
            const unsigned byte = (r << 4) | c;
            if (head > 0) {
                *dst++ = (uint8_t)byte;
                --head;
            } else {
                buf |= (unsigned long long)byte << (8 * nb);
                if (++nb == 8) {
                    *reinterpret_cast<unsigned long long*>(dst) = buf;
                    dst += 8;
                    buf = 0;
                    nb = 0;
                }
            }
        }
    }
    for (int i = 0; i < nb; ++i) dst[i] = (uint8_t)(buf >> (8 * i));
}

// =========================================================================================
// Default mapping of steps 2 and 3.
//   step 2: one thread per (A tile, B tile) PAIR.  The C tile mask is an OR over the tile's pairs,
//           and OR is associative, so the pairs are the unit of work: no thread waits on a long
//           pair list (hub tiles own thousands of pairs), every lane of every warp owns one 16x16
//           boolean product.
//   step 3: step3.cu.
// =========================================================================================

// first tile of every PEM_PAIR_BLOCK-pair step-2 block (every C' tile owns >= 1 pair, so a block overlaps
// at most PEM_PAIR_BLOCK + 1 tiles)
constexpr int S2P_THREADS = PEM_PAIR_BLOCK;
__global__ void __launch_bounds__(256)
k_pairblock_tiles(int64_t n_tiles, const int64_t* __restrict__ pair_ptr, int32_t* __restrict__ blk_tile)
{
    int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_tiles) return;
    const int64_t s = pair_ptr[t], e = pair_ptr[t + 1];
    for (int64_t b = (s + S2P_THREADS - 1) / S2P_THREADS; b * S2P_THREADS < e; ++b) blk_tile[b] = (int32_t)t;
}

// step 2, kernel 1 (pair-owner).  Lane = pair:
//   prod[r] = OR over k in Arow[r] of Bmask[k]             (16x16 boolean product)
//   hit     = (rows with prod != 0) << 16 | (OR of prod)    which C rows / columns the pair touches
// The lane walks the A tile's nonzero list ((r<<4)|k bytes, the reference's *tiles_rowColIdx): one
// 2-byte B mask load and one shared-memory OR per A nonzero, no per-row loops, so a warp's trip
// count is the largest A tile among its 32 pairs instead of 16 x the largest row.
// The hit words of 32 consecutive pairs are bit-transposed (5 butterfly shuffles) and stored as one
// 32-word block: word 16+r (resp. c) of block b has bit i set iff pair 32b+i touches C row r
// (resp. column c).  Step 3 ANDs two of those words to find the pairs feeding an entry (r, c)
// without walking the list.
// The products of a tile's pairs are OR-reduced by a segmented warp scan (pairs of a tile are
// consecutive lanes); a run that lies inside one warp is stored, a run cut by a warp boundary is
// merged with atomicOr into the zero-initialised mask array.
//
// ROWS = true (dense tiles: stencil / FEM operands, chosen on the host from nnz(A) / tiles(A)): the same product
// from the ROW MASKS alone.  The lane loads A's sixteen row masks and B's sixteen row masks with two 128-bit
// loads each (one 32-byte sector per tile: no nonzero list, no value offsets, no 1- and 2-byte gathers), parks
// B's rows in its own shared-memory column (conflict-free, read back only by the lane that wrote them) and
// forms prod[rows 2w, 2w+1] in a REGISTER per A mask word: one shared-memory load per A nonzero, nothing else
// touches the load/store unit (the list form was bound by it: 91 % of the L1 throughput on config 4).
// HITS = false (dense-tile mode: row form and step 3 is going to be the window kernel, which finds its pairs in shared
// memory): no hit words, no transposes, nothing stored per pair.
template <bool ROWS, bool HITS>
__global__ void __launch_bounds__(S2P_THREADS, 2048 / S2P_THREADS)
k_step2_pairs(int64_t n_pairs, int64_t n_tiles, const int32_t* __restrict__ blk_tile,
              const int64_t* __restrict__ pair_ptr, const int2* __restrict__ pairs,
              const uint32_t* __restrict__ A_off, const uint8_t* __restrict__ A_rc,
              const uint16_t* __restrict__ A_masks_t, const uint16_t* __restrict__ Amasks,
              const uint32_t* __restrict__ B_off, const uint8_t* __restrict__ B_rc,
              const uint16_t* __restrict__ Bmasks,
              uint32_t* __restrict__ Cmasks32, uint32_t* __restrict__ hit_t)
{
    __shared__ int s_ptr[S2P_THREADS + 2];
    // list form: word w of thread t at [w * THREADS + t]; row form: B's row k of thread t at [k * THREADS + t] (conflict-free)
    __shared__ unsigned s_acc[(ROWS ? 16 : 8) * S2P_THREADS];
    const int tid = threadIdx.x, lane = tid & 31;
    const int64_t i0 = (int64_t)blockIdx.x * S2P_THREADS;
    const int64_t t_lo = blk_tile[blockIdx.x];
    const int64_t t_hi = (i0 + S2P_THREADS < n_pairs) ? (int64_t)blk_tile[blockIdx.x + 1] : n_tiles - 1;
    const int span = (int)(t_hi - t_lo) + 1;
    for (int x = tid; x <= span; x += S2P_THREADS) {
        const int64_t rel = pair_ptr[t_lo + x] - i0;
        s_ptr[x] = (int)max((int64_t)-0x40000000, min(rel, (int64_t)0x40000000));
    }
    if (!ROWS) {
#pragma unroll
        for (int w = 0; w < 8; ++w) s_acc[w * S2P_THREADS + tid] = 0u;
    }
    __syncthreads();
    const int64_t i = i0 + tid;
    const bool valid = i < n_pairs;
    int x = 0;
    if (valid) {                                    // last x with s_ptr[x] <= tid
        int lo = 0, hi = span - 1;
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (s_ptr[mid] <= tid) lo = mid; else hi = mid - 1;
        }
        x = lo;
    }
    const int seg_s = valid ? s_ptr[x] : tid, seg_e = valid ? s_ptr[x + 1] : tid + 1;   // run of this tile, block-relative
    // Two ways to form the product, chosen per pair by the shorter nonzero list:
    //   by A's nonzeros (r,k):  prod[r] |= Bmask[k]                 (shared-memory OR, one per A nonzero)
    //   by B's nonzeros (k,c):  prod[r] |= 1 << c for r in AcolMask[k]   (registers; a hub A tile times
    //                           an ordinary B tile costs 1-2 steps instead of up to 256)
    unsigned acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    bool by_b = false;
    if (ROWS) {
        if (valid) {
            const int2 ab = pairs[i];
            const uint4* __restrict__ a4 = reinterpret_cast<const uint4*>(Amasks + (size_t)(unsigned)ab.x * 16u);
            const uint4* __restrict__ b4 = reinterpret_cast<const uint4*>(Bmasks + (size_t)(unsigned)ab.y * 16u);
            const uint4 ax = a4[0], ay = a4[1], bx = b4[0], by = b4[1];
            const unsigned bw[8] = {bx.x, bx.y, bx.z, bx.w, by.x, by.y, by.z, by.w};
            unsigned* my = s_acc + tid;
#pragma unroll
            for (int w = 0; w < 8; ++w) {               // B row k of this pair at my[k * THREADS]
                my[(2 * w) * S2P_THREADS] = bw[w] & 0xFFFFu;
                my[(2 * w + 1) * S2P_THREADS] = bw[w] >> 16;
            }
            const unsigned aw[8] = {ax.x, ax.y, ax.z, ax.w, ay.x, ay.y, ay.z, ay.w};
#pragma unroll
            for (int w = 0; w < 8; ++w) {               // word w = rows 2w (low half), 2w + 1 (high half)
                unsigned m = aw[w] & 0xFFFFu, p = 0, q = 0;
                while (m) {                             // prod[2w] = OR over k in Arow[2w] of Brow[k]: eight instructions per nonzero
                    const unsigned k = __ffs(m) - 1u;
                    m &= m - 1u;
                    p |= my[k * S2P_THREADS];
                }
                m = aw[w] >> 16;
                while (m) {
                    const unsigned k = __ffs(m) - 1u;
                    m &= m - 1u;
                    q |= my[k * S2P_THREADS];
                }
                acc[w] = p | (q << 16);
            }
        }
    } else if (valid) {
        const int2 ab = pairs[i];
        const uint32_t a0 = A_off[ab.x], a1 = A_off[ab.x + 1];
        const uint32_t b0 = B_off[ab.y], b1 = B_off[ab.y + 1];
        by_b = 8u * (b1 - b0) < (a1 - a0);      // ~48 instructions per B nonzero against ~16 per A nonzero, and a warp pays for both paths
        if (by_b) {
            const uint16_t* __restrict__ at = A_masks_t + (size_t)(unsigned)ab.x * 16u;
            for (uint32_t e = b0; e < b1; ++e) {
                const unsigned kc = B_rc[e];
                const unsigned rows = at[kc >> 4];           // rows of A holding column k
                const unsigned c = kc & 15u;
#pragma unroll
                for (int w = 0; w < 8; ++w) {
                    const unsigned two = (rows >> (2 * w)) & 3u;          // rows 2w, 2w+1
                    acc[w] |= ((two & 1u) | ((two & 2u) << 15)) << c;
                }
            }
        } else {
            const uint16_t* __restrict__ bm = Bmasks + (size_t)(unsigned)ab.y * 16u;
            unsigned* my = s_acc + tid;
#pragma unroll 2
            for (uint32_t e = a0; e < a1; ++e) {
                const unsigned rc = A_rc[e];
                const unsigned o = bm[rc & 15u];
                const unsigned r = rc >> 4;
                my[(r >> 1) * S2P_THREADS] |= o << ((r & 1u) * 16u);
            }
        }
    }
    if (!ROWS && !by_b) {
#pragma unroll
        for (int w = 0; w < 8; ++w) acc[w] = s_acc[w * S2P_THREADS + tid];
    }
    if (HITS) {
        unsigned hit = 0;
        {
            unsigned c = 0, rows_hit = 0;
#pragma unroll
            for (int w = 0; w < 8; ++w) {
                c |= acc[w];
                rows_hit |= ((acc[w] & 0xFFFFu) ? 1u : 0u) << (2 * w);
                rows_hit |= ((acc[w] >> 16) ? 1u : 0u) << (2 * w + 1);
            }
            hit = (rows_hit << 16) | ((c | (c >> 16)) & 0xFFFFu);
        }
        // 32x32 bit transpose across the warp: afterwards lane b holds bit b of every lane's hit word
        unsigned v = hit, m = 0x0000FFFFu;
#pragma unroll
        for (int j = 16; j > 0; j >>= 1) {
            const unsigned y = __shfl_xor_sync(0xffffffffu, v, j);
            v = (lane & j) ? ((v & ~m) | ((y >> j) & m)) : ((v & ~(m << j)) | ((y & m) << j));
            m ^= m << (j >> 1);
        }
        if (i0 + (tid & ~31) < n_pairs) hit_t[i0 + tid] = v;
    }
    // segmented inclusive OR scan along the lanes of a tile's run
    const int wfirst = tid & ~31;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const bool take = lane >= o && tid - o >= seg_s;
        if (!__any_sync(0xffffffffu, take)) break;
#pragma unroll
        for (int w = 0; w < 8; ++w) {
            const unsigned v = __shfl_up_sync(0xffffffffu, acc[w], o);
            acc[w] |= take ? v : 0u;
        }
    }
    const bool tail = valid && (lane == 31 || tid + 1 >= seg_e);
    if (tail) {
        uint32_t* out = Cmasks32 + (size_t)(t_lo + x) * 8;
        if (seg_s >= wfirst && seg_e <= wfirst + 32) {
            reinterpret_cast<uint4*>(out)[0] = make_uint4(acc[0], acc[1], acc[2], acc[3]);
            reinterpret_cast<uint4*>(out)[1] = make_uint4(acc[4], acc[5], acc[6], acc[7]);
        } else {
#pragma unroll
            for (int w = 0; w < 8; ++w)
                if (acc[w]) atomicOr(&out[w], acc[w]);
        }
    }
}

// step 2, kernel 1, alternative mapping (PEM_OPT_STEP2_KERNEL = 2; an independent formulation the tests
// cross-check the pair kernel with): SIXTEEN LANES PER C' TILE, lane = row r, the tile's pairs walked in order.  Per pair the half-warp loads
// A's 16 row masks and B's 16 row masks with one coalesced 32-byte load each; lane r then ORs B's row k for
// every k in Arow[r], fetching it from the lane that holds it with a shuffle: no nonzero list, no shared
// memory, no per-nonzero gather, and the trip count of a pair is the longest A row (3 for a band) instead
// of the A tile's nonzero count.  The pair's hit word (C rows touched << 16 | C columns touched) comes
// from one ballot and one OR-reduction; k_hit_transpose turns 32 consecutive hit words into step 3's
// bit-transposed block afterwards.
__global__ void __launch_bounds__(256)
k_step2_tiles(int64_t n_tiles, const int64_t* __restrict__ pair_ptr, const int2* __restrict__ pairs,
              const uint16_t* __restrict__ Amasks, const uint16_t* __restrict__ Bmasks,
              uint16_t* __restrict__ Cmasks, uint32_t* __restrict__ hit)
{
    const int tid = threadIdx.x;
    const int64_t t = ((int64_t)blockIdx.x * blockDim.x + tid) >> 4;
    const unsigned r = tid & 15u;
    if (t >= n_tiles) return;                       // whole 16-lane groups leave together
    const unsigned sh = tid & 16u;
    const unsigned grp = 0xFFFFu << sh;
    const int64_t ps = pair_ptr[t];
    const unsigned np = (unsigned)(pair_ptr[t + 1] - ps);
    const int2* __restrict__ pl = pairs + ps;
    uint32_t* __restrict__ hp = hit + ps;
    unsigned acc = 0;
    int2 ab = pl[0];
    unsigned am = Amasks[(size_t)(unsigned)ab.x * 16u + r], bm = Bmasks[(size_t)(unsigned)ab.y * 16u + r];
    for (unsigned i = 0; i < np; ++i) {
        unsigned a = am;
        const unsigned b = bm;
        if (i + 1 < np) {                           // next pair's masks while this one is consumed
            ab = pl[i + 1];
            am = Amasks[(size_t)(unsigned)ab.x * 16u + r];
            bm = Bmasks[(size_t)(unsigned)ab.y * 16u + r];
        }
        unsigned p = 0;
        while (__any_sync(grp, a != 0)) {           // uniform over the sixteen lanes: every lane feeds the shuffle
            const unsigned k = a ? (unsigned)__ffs(a) - 1u : 0u;
            const unsigned v = __shfl_sync(grp, b, (int)k, 16);
            p |= a ? v : 0u;
            a &= a - 1u;
        }
        acc |= p;
        const unsigned rows_hit = (__ballot_sync(grp, p != 0) >> sh) & 0xFFFFu;
        const unsigned cols_hit = __reduce_or_sync(grp, p);
        if (r == 0) hp[i] = (rows_hit << 16) | cols_hit;
    }
    Cmasks[t * 16 + r] = (uint16_t)acc;
}

// hit words of 32 consecutive pairs -> one bit-transposed 32-word block, in place (what k_step2_pairs
// produces directly): afterwards word 16+r (resp. c) of block b has bit i set iff pair 32b+i touches C row
// r (resp. column c)
__global__ void __launch_bounds__(256)
k_hit_transpose(int64_t n_pairs, uint32_t* __restrict__ hit)
{
    const int lane = threadIdx.x & 31;
    const int64_t base = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) & ~(int64_t)31;
    if (base >= n_pairs) return;                    // whole warps leave together
    unsigned v = base + lane < n_pairs ? hit[base + lane] : 0u, m = 0x0000FFFFu;
#pragma unroll
    for (int j = 16; j > 0; j >>= 1) {
        const unsigned y = __shfl_xor_sync(0xffffffffu, v, j);
        v = (lane & j) ? ((v & ~m) | ((y >> j) & m)) : ((v & ~(m << j)) | ((y & m) << j));
        m ^= m << (j >> 1);
    }
    hit[base + lane] = v;                           // the array is padded to whole blocks
}

// per-tile nnz = popcount of the 256-bit mask, fed straight into the exclusive scan
struct TileNnz {
    const uint4* masks;
    int64_t n_tiles;
    __device__ __forceinline__ int64_t operator()(int64_t t) const
    {
        if (t >= n_tiles) return 0;
        const uint4 a = masks[2 * t], b = masks[2 * t + 1];
        return __popc(a.x) + __popc(a.y) + __popc(a.z) + __popc(a.w) + __popc(b.x) + __popc(b.y) + __popc(b.z) + __popc(b.w);
    }
};

__global__ void k_set_last_i64(int64_t* p, int64_t idx, int64_t v) { p[idx] = v; }

}  // namespace

// =========================================================================================
// host side
// =========================================================================================
static int check_operands(pem_ctx* ctx, const pem_tiled* A, const pem_tiled* B, int rb, int re)
{
    if (!ctx || !A || !B) return PEM_ERR_ARG;
    if (A->cols != B->rows) return ctx->fail(PEM_ERR_ARG, "inner dimensions differ (A.cols != B.rows)");
    if (rb < 0 || re < rb || re > A->tile_rows) return ctx->fail(PEM_ERR_ARG, "tile-row panel out of range");
    return PEM_OK;
}

extern "C" {

int pem_step2_symbolic(pem_ctx* ctx, const pem_tiled* A, const pem_tiled* B, pem_result* C)
{
    PEM_RANGE("pem_step2_symbolic");
    if (!ctx || !A || !B || !C) return PEM_ERR_ARG;
    if (C->stage != 1) return ctx->fail(PEM_ERR_ARG, "step 2 needs a result fresh from step 1");
    if (C->tiles >= 0x7fffffffLL)
        return ctx->fail(PEM_ERR_LIMIT, "more than 2^31 C' tiles in one result: multiply in tile-row panels (pem_spgemm_panel)");
    const bool rows_variant = ctx->opt_owner == 1;
    if (C->dtype == PEM_F32 && (rows_variant || ctx->opt_owner == 3))
        return ctx->fail(PEM_ERR_ARG, "fp32 products run the default kernels only (PEM_OPT_OWNER 0 / 2 / 4)");
    const int64_t nblk = (C->pairs + S2P_THREADS - 1) / S2P_THREADS;
    if (!rows_variant && nblk > 0x7fffffffLL) return ctx->fail(PEM_ERR_LIMIT, "more than 2^39 tile pairs");
    PEM_CK(cudaSetDevice(ctx->device));
    // buffers of an earlier call that failed part-way: a retry must not overwrite live blocks
    pem_free(ctx, C->masks); pem_free(ctx, C->tile_nnz_ptr); pem_free(ctx, C->pair_hit);
    PEM_TRY(pem_alloc(ctx, &C->masks, (size_t)C->tiles * 16));
    PEM_TRY(pem_alloc(ctx, &C->tile_nnz_ptr, (size_t)C->tiles + 1));
    if (rows_variant) {
        if (C->tiles > 0) {
            k_step2_masks<<<pem_div_up(C->tiles * 16, 256), 256, 0, ctx->stream>>>(
                C->tiles, C->pair_ptr, C->pair_list, A->masks, B->masks, C->masks, C->tile_nnz_ptr);
            PEM_LAUNCHED();
        }
        k_set_last_i64<<<1, 1, 0, ctx->stream>>>(C->tile_nnz_ptr, C->tiles, 0);
        PEM_LAUNCHED();
        PEM_TRY(pem_scan_exclusive_i64(ctx, C->tile_nnz_ptr, C->tiles + 1));
    } else {
        // one lane per pair by default; sixteen lanes per C' tile (k_step2_tiles) on request: measured on B200 it
        // loses even on the stencil product it was written for (config 4: 7.1 ms against 3.4 ms)
        const bool by_tiles = ctx->opt_step2_kernel == 2;
        // row form for dense tiles (at least eight nonzeros per A tile on average; config 4: 17.9), list form otherwise
        // (hypersparse tiles: one or two list steps per pair; hub tiles walk the shorter of the two lists)
        const bool rows_form = ctx->opt_step2_kernel == 3 ||
                               (ctx->opt_step2_kernel == 0 && A->nnz >= 8 * (int64_t)A->tiles);
        // dense-tile mode: both operands' tiles are dense and the numeric kernel is left to the engine (or is the window
        // kernel): step 3 will run the window kernel, whose pairs sit in shared memory, so the per-pair hit words (a
        // ninth of this kernel's instructions and 4 bytes per pair) are not produced at all
        const bool hits = !(ctx->opt_step2_kernel == 0 && rows_form && !by_tiles && (ctx->opt_owner == 0 || ctx->opt_owner == 4) &&
                            B->nnz >= 8 * (int64_t)B->tiles);
        if (hits) PEM_TRY(pem_alloc(ctx, &C->pair_hit, (size_t)nblk * S2P_THREADS));
        if (by_tiles && C->pairs > 0) {
            pem_free(ctx, C->pair_blk);
            KT_BEGIN(KT_PAIRS);
            k_step2_tiles<<<pem_div_up(C->tiles * 16, 256), 256, 0, ctx->stream>>>(
                C->tiles, C->pair_ptr, C->pair_list, A->masks, B->masks, C->masks, C->pair_hit);
            PEM_LAUNCHED();
            k_hit_transpose<<<pem_div_up(C->pairs, 256), 256, 0, ctx->stream>>>(C->pairs, C->pair_hit);
            KT_END(KT_PAIRS);
            PEM_LAUNCHED();
        } else if (C->pairs > 0) {
            PEM_CK(cudaMemsetAsync(C->masks, 0, (size_t)C->tiles * 32, ctx->stream));
            int32_t* blk = C->pair_blk;            // expand-sort-compress leaves it behind (k_ctiles)
            C->pair_blk = nullptr;
            pem_guard g(ctx, blk);
            if (!blk) {
                PEM_TRY(pem_alloc(ctx, &blk, (size_t)nblk + 1));
                k_pairblock_tiles<<<pem_div_up(C->tiles, 256), 256, 0, ctx->stream>>>(C->tiles, C->pair_ptr, blk);
                PEM_LAUNCHED();
            }
            KT_BEGIN(KT_PAIRS);
#define S2P_ARGS C->pairs, C->tiles, blk, C->pair_ptr, C->pair_list, A->tile_nnz_ptr, A->rc_idx, A->masks_t, A->masks, \
                B->tile_nnz_ptr, B->rc_idx, B->masks, reinterpret_cast<uint32_t*>(C->masks), C->pair_hit
            if (rows_form && !hits) k_step2_pairs<true, false><<<(unsigned)nblk, S2P_THREADS, 0, ctx->stream>>>(S2P_ARGS);
            else if (rows_form) k_step2_pairs<true, true><<<(unsigned)nblk, S2P_THREADS, 0, ctx->stream>>>(S2P_ARGS);
            else k_step2_pairs<false, true><<<(unsigned)nblk, S2P_THREADS, 0, ctx->stream>>>(S2P_ARGS);
#undef S2P_ARGS
            KT_END(KT_PAIRS);
            PEM_LAUNCHED();
            pem_free(ctx, blk);
        } else {
            PEM_CK(cudaMemsetAsync(C->masks, 0, (size_t)C->tiles * 32, ctx->stream));
        }
        // per-tile nnz (popcount of the mask) -> exclusive scan, in one pass over the masks
        auto nnz_it = thrust::make_transform_iterator(thrust::counting_iterator<int64_t>(0),
                                                      TileNnz{reinterpret_cast<const uint4*>(C->masks), C->tiles});
        size_t tb = 0;
        PEM_CK(cub::DeviceScan::ExclusiveSum(nullptr, tb, nnz_it, C->tile_nnz_ptr, C->tiles + 1, ctx->stream));
        char* tmp = nullptr;
        pem_guard g(ctx, tmp);
        PEM_TRY(pem_alloc(ctx, &tmp, tb));
        PEM_CK(cub::DeviceScan::ExclusiveSum(tmp, tb, nnz_it, C->tile_nnz_ptr, C->tiles + 1, ctx->stream));
        ctx->launches += 2;
        pem_free(ctx, tmp);
    }
    {
        pem_size_read rd(ctx);
        PEM_TRY(rd.add(C->tile_nnz_ptr + C->tiles, 1));
        PEM_TRY(rd.get(&C->nnz));
    }
    C->stage = 2;
    C->s2_pairs = !rows_variant;
    // step-3 mapping (step3.cu): the entry-owner kernel unless the tile-class kernel is asked for
    C->s3_entries = ctx->opt_owner != 3;
    return PEM_OK;
}

// Ctiles_rowColIdx on demand (see k_rowcolidx)
int pem_result_make_rowcolidx(pem_ctx* ctx, pem_result* C)
{
    if (!ctx || !C) return PEM_ERR_ARG;
    if (C->stage < 2) return ctx->fail(PEM_ERR_ARG, "rowColIdx needs step 2");
    if (C->row_col_idx) return PEM_OK;
    PEM_CK(cudaSetDevice(ctx->device));
    PEM_TRY(pem_alloc(ctx, &C->row_col_idx, (size_t)C->nnz));
    if (C->tiles > 0) {
        k_rowcolidx<<<pem_div_up(C->tiles, 128), 128, 0, ctx->stream>>>(C->tiles, C->masks, C->tile_nnz_ptr, C->row_col_idx);
        PEM_LAUNCHED();
    }
    return PEM_OK;
}

// a result whose buffers went back to the allocator behind its back (abandoned graph capture): drop the pointers
static void result_forget_buffers(pem_result* C)
{
    for (void** f : C->buffers()) *f = nullptr;
}

// hand every block of an abandoned (or over-budget) graph arena back to ordinary ownership: `keep` are the
// pointers a live result still uses (they stay live blocks of the context), the rest goes to the cache
static void graph_dissolve(pem_ctx* ctx, pem_graph* g, pem_result* keep)
{
    std::unordered_set<const void*> held;
    if (keep)
        for (void** f : keep->buffers()) if (*f) held.insert(*f);
    for (auto& b : g->arena)
        if (!held.count(b.first) && ctx->live_blocks.count(b.first)) pem_free_bytes(ctx, b.first);
    g->arena.clear(); g->owned.clear(); g->idle.clear(); g->bytes = 0;
    if (g->exec) { cudaGraphExecDestroy(g->exec); g->exec = nullptr; }
}

int pem_spgemm_panel(pem_ctx* ctx, const pem_tiled* A, const pem_tiled* B,
                     int32_t rb, int32_t re, pem_result** out, pem_times* times)
{
    PEM_RANGE("pem_spgemm_panel");
    if (!out) return PEM_ERR_ARG;
    *out = nullptr;
    PEM_TRY(check_operands(ctx, A, B, rb, re));
    PEM_CK(cudaSetDevice(ctx->device));
    PEM_CK(cudaStreamSynchronize(ctx->stream));
    auto w0 = std::chrono::high_resolution_clock::now();
    pem_result* C = nullptr;
    // size plan of this (A, B, panel): recorded by the first product, replayed (no host stall before the final
    // synchronisation) by every later one
    const std::vector<int64_t> key = {(int64_t)A->uid, (int64_t)B->uid, rb, re, ctx->opt_keep_empty, ctx->opt_step1_path,
                                      ctx->opt_esc_variant};
    // the three steps, enqueued on the context's stream (or captured from it)
    auto run_steps = [&]() -> int {
        PEM_CK(pem_event_record(ctx, ctx->ev[2]));
        PEM_TRY(pem_step1_symbolic(ctx, A, B, rb, re, &C));
        pem_event_record(ctx, ctx->ev[3]);
        PEM_TRY(pem_step2_symbolic(ctx, A, B, C));
        pem_event_record(ctx, ctx->ev[4]);
        PEM_TRY(pem_step3_numeric(ctx, A, B, C));
        pem_event_record(ctx, ctx->ev[5]);
        return PEM_OK;
    };
    int redo = 0;
    for (;;) {
        ctx->plan = nullptr;
        ctx->plan_replay = false;
        ctx->plan_pos = 0;
        pem_plan* plan = nullptr;
        if (ctx->opt_plans) {
            if (ctx->plans.size() > 256) ctx->plans.clear();
            plan = &ctx->plans[key];
            ctx->plan = plan;
            ctx->plan_replay = plan->valid;
        }
        for (int i = 0; i < KT_N; ++i) { ctx->kt_seen[i] = false; ctx->kt_ms[i] = 0.0; }
        // Product graph (PEM_OPT_GRAPHS): the second product of a plan is CAPTURED from the stream while the host code
        // below replays the plan (so it never stalls), then launched; later products launch the same graph.
        int gopts[5];
        pem_graph_opts(ctx, gopts);
        // (one graph may hold at most an eighth of the graphs' memory budget: where a product moves gigabytes, its
        //  launches are not what it waits for, and sequential panels of a large product must not park their buffers)
        const bool graph_ok = plan && plan->valid && ctx->opt_graphs && !plan->graph_failed && !ctx->opt_trace &&
                              !A->vals_pending && !B->vals_pending &&
                              (plan->graph || plan->alloc_bytes <= ctx->graph_limit / 8);
        ctx->prod_alloc = 0;
        std::shared_ptr<pem_graph> g;
        bool launch_only = false, capture = false;
        if (graph_ok && plan->graph) {
            launch_only = !plan->graph->busy && std::equal(gopts, gopts + 5, plan->graph->opts);
            if (launch_only) g = plan->graph;
        } else if (graph_ok) {
            g = std::make_shared<pem_graph>();
            std::copy(gopts, gopts + 5, g->opts);
            if (cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeRelaxed) == cudaSuccess) {
                capture = true;
                ctx->cap = g.get();
            } else {
                (void)cudaGetLastError();
                plan->graph_failed = true;
                g.reset();
            }
        }
        int rc = PEM_OK;
        if (launch_only) {
            cudaError_t e = cudaGraphLaunch(g->exec, ctx->stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
            if (e != cudaSuccess) rc = ctx->fail_cuda(e, "launch of a product graph", __FILE__, __LINE__);
            else {
                C = new pem_result(g->tmpl);
                C->graph = g;
                g->busy = true;
                ctx->launches += g->launches;
                ctx->last_step3_kernel = g->last_step3_kernel;
                ctx->last_sort_passes = g->last_sort_passes;
                for (int i = 0; i < KT_N; ++i) ctx->kt_seen[i] = g->kt_seen[i];
                ctx->plan_pos = plan->n;
                ++ctx->graph_replays;
            }
        } else if (capture) {
            const int64_t launches0 = ctx->launches;
            rc = run_steps();
            ctx->cap = nullptr;
            cudaGraph_t gr = nullptr;
            cudaError_t e = cudaStreamEndCapture(ctx->stream, &gr);
            if (rc == PEM_OK && e == cudaSuccess && gr) e = cudaGraphInstantiate(&g->exec, gr, 0);
            if (gr) cudaGraphDestroy(gr);
            if (rc == PEM_OK && e == cudaSuccess && g->exec && g->side_allocs) e = cudaStreamSynchronize(ctx->copy_stream);
            if (rc == PEM_OK && e == cudaSuccess && g->exec) e = cudaGraphLaunch(g->exec, ctx->stream);
            if (rc == PEM_OK && e == cudaSuccess && g->exec) e = cudaStreamSynchronize(ctx->stream);
            if (rc != PEM_OK || e != cudaSuccess || !g->exec) {
                // not capturable (a host stall or an unsupported call inside), or the launch failed: give the blocks
                // back, remember not to try again, and run this product the ordinary way
                (void)cudaGetLastError();
                (void)cudaStreamSynchronize(ctx->stream);
                (void)cudaGetLastError();
                graph_dissolve(ctx, g.get(), nullptr);
                if (C) { result_forget_buffers(C); delete C; C = nullptr; }
                ctx->launches = launches0;              // nothing of the abandoned capture ran
                plan->graph_failed = true;
                ctx->err.clear();
                ctx->plan = nullptr;
                ctx->plan_replay = false;
                continue;
            }
            g->ctx = ctx;
            g->launches = ctx->launches - launches0;
            g->last_step3_kernel = ctx->last_step3_kernel;
            g->last_sort_passes = ctx->last_sort_passes;
            for (int i = 0; i < KT_N; ++i) g->kt_seen[i] = ctx->kt_seen[i];
            ++ctx->graph_replays;
            if (ctx->graph_bytes + g->bytes <= ctx->graph_limit) {
                g->tmpl = *C;
                C->graph = g;
                g->busy = true;
                plan->graph = g;
                ctx->graph_bytes += g->bytes;
            } else {                                    // over the budget: this product keeps its buffers as an ordinary result
                g->ctx = nullptr;
                graph_dissolve(ctx, g.get(), C);
                plan->graph_failed = true;
            }
        } else {
            rc = run_steps();
            if (rc == PEM_OK && cudaStreamSynchronize(ctx->stream) != cudaSuccess)
                rc = ctx->fail_cuda(cudaGetLastError(), "cudaStreamSynchronize after step 3", __FILE__, __LINE__);
        }
        pem_plan* pl = ctx->plan;
        const bool replayed = ctx->plan_replay;
        const int npos = ctx->plan_pos;
        ctx->plan = nullptr;
        ctx->plan_replay = false;
        if (rc != PEM_OK) {
            pem_result_free(ctx, C);
            if (pl) ctx->plans.erase(key);
            return rc;
        }
        if (!pl) break;
        if (!replayed) {
            pl->n = npos;
            pl->valid = true;
            pl->alloc_bytes = ctx->prod_alloc;
            break;
        }
        bool same = npos == pl->n;
        for (int i = 0; same && i < npos; ++i) same = ctx->h_check[i] == pl->v[i];
        if (same) break;
        pem_result_free(ctx, C);                    // never expected: redo the product with the stalls
        C = nullptr;
        ctx->plans.erase(key);
        if (++redo == 2) return ctx->fail(PEM_ERR_CUDA, "sizes changed under a replayed size plan");
    }
    auto w1 = std::chrono::high_resolution_clock::now();
    for (int i = 0; i < KT_N; ++i) {
        float ms = 0.f;
        if (ctx->kt_seen[i] && cudaEventElapsedTime(&ms, ctx->kev[2 * i], ctx->kev[2 * i + 1]) == cudaSuccess) ctx->kt_ms[i] = ms;
        else (void)cudaGetLastError();
    }
    if (times) {
        float s1 = 0, s2 = 0, s3 = 0;
        if (cudaEventElapsedTime(&s1, ctx->ev[2], ctx->ev[3]) != cudaSuccess) { s1 = 0; (void)cudaGetLastError(); }
        if (cudaEventElapsedTime(&s2, ctx->ev[3], ctx->ev[4]) != cudaSuccess) { s2 = 0; (void)cudaGetLastError(); }
        if (cudaEventElapsedTime(&s3, ctx->ev[4], ctx->ev[5]) != cudaSuccess) { s3 = 0; (void)cudaGetLastError(); }
        times->step1_ms = s1; times->step2_ms = s2; times->step3_ms = s3;
        times->kernel_ms = (double)s1 + s2 + s3;
        times->total_ms = std::chrono::duration<double, std::milli>(w1 - w0).count();
        times->malloc_ms = times->total_ms - times->kernel_ms;
    }
    *out = C;
    return PEM_OK;
}

int pem_spgemm(pem_ctx* ctx, const pem_tiled* A, const pem_tiled* B, pem_result** C, pem_times* times)
{
    if (!A) return PEM_ERR_ARG;
    return pem_spgemm_panel(ctx, A, B, 0, A->tile_rows, C, times);
}

// Step 3 again on a complete result, from the operands' current values: the kernel C's own step 3 ran (the choice
// PEM_OPT_OWNER made then is baked into C: a dense-tile-mode result has no hit words for any other kernel), on C's
// buffers, with no size read-back.  A result borrowed from a product graph is fine: the graph does not run while
// the result is alive.
int pem_spgemm_numeric(pem_ctx* ctx, const pem_tiled* A, const pem_tiled* B, pem_result* C, pem_times* times)
{
    PEM_RANGE("pem_spgemm_numeric");
    if (!ctx || !A || !B || !C) return PEM_ERR_ARG;
    if (C->stage != 3) return ctx->fail(PEM_ERR_ARG, "pem_spgemm_numeric needs a complete result (step 3 done)");
    if (C->a_uid != A->uid || C->b_uid != B->uid)
        return ctx->fail(PEM_ERR_ARG, "pem_spgemm_numeric: A and B are not the handles the result was computed from");
    if (A->dtype != C->dtype || B->dtype != C->dtype) return ctx->fail(PEM_ERR_ARG, "operands and result have different value types");
    PEM_CK(cudaSetDevice(ctx->device));
    PEM_CK(cudaStreamSynchronize(ctx->stream));
    auto w0 = std::chrono::high_resolution_clock::now();
    PEM_TRY(pem_tiled_wait_vals(ctx, A));
    PEM_TRY(pem_tiled_wait_vals(ctx, B));
    for (int i = 0; i < KT_N; ++i) { ctx->kt_seen[i] = false; ctx->kt_ms[i] = 0.0; }
    PEM_CK(pem_event_record(ctx, ctx->ev[4]));
    PEM_TRY(pem_step3_launch(ctx, A, B, C));
    PEM_CK(pem_event_record(ctx, ctx->ev[5]));
    PEM_CK(cudaStreamSynchronize(ctx->stream));
    ctx->last_step3_kernel = C->s3_kernel;
    auto w1 = std::chrono::high_resolution_clock::now();
    float ms = 0.f;
    if (ctx->kt_seen[KT_NUMERIC] && cudaEventElapsedTime(&ms, ctx->kev[2 * KT_NUMERIC], ctx->kev[2 * KT_NUMERIC + 1]) == cudaSuccess)
        ctx->kt_ms[KT_NUMERIC] = ms;
    else
        (void)cudaGetLastError();
    if (times) {
        float s3 = 0.f;
        if (cudaEventElapsedTime(&s3, ctx->ev[4], ctx->ev[5]) != cudaSuccess) { s3 = 0.f; (void)cudaGetLastError(); }
        times->step1_ms = 0; times->step2_ms = 0; times->step3_ms = s3;
        times->kernel_ms = s3;
        times->total_ms = std::chrono::duration<double, std::milli>(w1 - w0).count();
        times->malloc_ms = times->total_ms - times->kernel_ms;
    }
    return PEM_OK;
}

}  // extern "C"
