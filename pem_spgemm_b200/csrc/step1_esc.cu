// Step 1, default path: tile-level symbolic SpGEMM by EXPAND - SORT - COMPRESS.
//
// Replaces, in /root/reference: tile_spgemm_step1_cuda_spa_kernel / ..._numeric_... (spgemm.cu:
// 271-384), the NSPARSE hash path chosen by `B_tileCols > 512*32` (spgemm.cu:1142,
// NSPARSE/spgemm_nsparse_kernel.h:1171-1438) and the CSC pair search
// pem_spgemm_step2_search_pairs (spgemm.cu:387-497).  Output contract as step1.cu: C' in CSR+COO
// with ascending tile columns, and per C' tile the (A tile, B tile) pairs in ascending k.
//
// The per-row accumulators of the reference (a 2 KB bitmap per warp, or hash tables binned by row
// length) serialise on hub rows: one tile row of a power-law matrix can own a third of all tile
// products.  Here the unit of work is the TILE PRODUCT, not the row:
//
//   products  k_tile_products: thread per A tile p: len(p) = |B' row of p's tile column|, and the
//             tile-column window [jmin, jmax] of every C' row (atomicMin/Max).  Exclusive scan of
//             len -> product index space [0, P).
//   split     k_merge_split: merge-path partition of (A tiles, products) into chunks of CHUNK
//             work items, so a block sees at most CHUNK tiles AND at most CHUNK products whatever
//             the row-length distribution (hub rows are cut across thousands of blocks).
//   expand    k_expand: a block stages its A-tile slice (product offsets, first B tile, column
//             occupancy, row) in shared memory; lanes take products warp-striped (coalesced 2-byte
//             rowOcc loads, 8 independent loads in flight per lane) and keep product (p, q) iff
//             colOcc(p) & rowOcc(q) != 0, i.e. iff the 16x16 boolean product of the two tiles is
//             non-empty.  Kept products are written in product order (ballot/popc ranks inside a
//             warp, a block scan across warps) as key = (C' row, tile column - jmin(row)),
//             value = (p, q).
//   compact   inside k_expand: the chunks' kept counts are chained by decoupled look-back while the kernel runs,
//             so every chunk writes straight to its final, compacted position (one pass over the pairs).
//   sort      ONE stable LSD radix sort of (key, value) over exactly the key bits in use.  Products
//             were emitted in ascending p, and p ascends with (row, k), so after a stable sort by
//             (row, column) every C' tile's pairs are contiguous and already in ascending k: the
//             order step 3 needs for bit-reproducible sums.
//   compress  heads of equal-key runs = C' tiles (stream compaction of run starts = pair_ptr);
//             k_ctiles decodes (row, col) and builds the CSR row pointer.
// No per-row shared-memory structure exists, so there is no limit on B's tile-column count and
// no long-row special case.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_select.cuh>
#include <thrust/iterator/counting_iterator.h>

#include <algorithm>
#include <climits>
#include <cstdlib>

#include <chrono>

#include "engine.cuh"

namespace {

// PEM_OPT_TRACE: host-side timeline of step 1 (where the host waits), printed to stderr
struct Trace {
    bool on;
    std::chrono::high_resolution_clock::time_point t0;
    explicit Trace(bool on_) : on(on_), t0(std::chrono::high_resolution_clock::now()) {}
    void mark(const char* what)
    {
        if (!on) return;
        auto t = std::chrono::high_resolution_clock::now();
        fprintf(stderr, "[step1 %8.3f ms] %s\n", std::chrono::duration<double, std::milli>(t - t0).count(), what);
    }
};

constexpr int EX_THREADS = 256;
constexpr int EX_ITEMS = 8;                       // products per lane
constexpr int EX_CHUNK = EX_THREADS * EX_ITEMS;   // work items (A tiles + products) per block
constexpr int EX_WARPS = EX_THREADS / 32;

// thread per A tile of the panel
__global__ void __launch_bounds__(256)
k_tile_products(int p0, int np, int rb, const int32_t* __restrict__ Acol, const int32_t* __restrict__ Arow,
                const uint16_t* __restrict__ AcolOcc,
                const int32_t* __restrict__ Brp, const int32_t* __restrict__ Bcol,
                const int64_t* __restrict__ srow_ptr,
                int64_t* __restrict__ plen, int32_t* __restrict__ bfirst, int64_t* __restrict__ icnt,
                int* __restrict__ jmin, int* __restrict__ jmax, int64_t* __restrict__ scalars)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long cost = 0, items = 0;
    int row = -1, lo = INT_MAX, hi = -1;
    if (i < np) {
        const int p = p0 + i;
        const int k = Acol[p];
        const int bs = Brp[k], be = Brp[k + 1];
        plen[i] = be - bs;
        bfirst[i] = bs;
        if (be > bs) {
            row = Arow[p] - rb;
            lo = Bcol[bs];
            hi = Bcol[be - 1];
        }
        if (srow_ptr) {            // cost of expanding this tile through B's row slices instead
            unsigned occ = AcolOcc[p];
            items = __popc(occ);
            icnt[i] = (int64_t)items;
            const int64_t* sp = srow_ptr + (size_t)k * 16;
            while (occ) {                       // per RUN of occupied columns: slices of consecutive rows are consecutive
                const int c = __ffs(occ) - 1;
                const int len = __ffs(~(occ >> c)) - 1;
                occ &= ~(((1u << len) - 1u) << c);
                cost += (unsigned long long)(sp[c + len] - sp[c]);
            }
        }
    } else if (i == np) {
        plen[i] = 0;
        if (srow_ptr) icnt[i] = 0;
    }
    {   // window of reachable tile columns per C' row: the tiles of a row are consecutive threads, so the
        // lanes of one row reduce among themselves and their leader issues the two atomics
        const unsigned peers = __match_any_sync(0xffffffffu, row);
        const int wlo = __reduce_min_sync(peers, lo), whi = __reduce_max_sync(peers, hi);
        if (row >= 0 && (threadIdx.x & 31) == __ffs(peers) - 1) {
            if (wlo < jmin[row]) atomicMin(&jmin[row], wlo);
            if (whi > jmax[row]) atomicMax(&jmax[row], whi);
        }
    }
    if (srow_ptr) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            cost += __shfl_xor_sync(0xffffffffu, cost, o);
            items += __shfl_xor_sync(0xffffffffu, items, o);
        }
        if ((threadIdx.x & 31) == 0 && items) {
            atomicAdd((unsigned long long*)&scalars[SC_T2], cost);
            atomicAdd((unsigned long long*)&scalars[SC_T1], items);
        }
    }
}

// row-sliced expansion: one work item per (A tile p, occupied tile column c of p); its products are
// the tiles of B's row slice 16*k + c.  A B tile reachable through several columns of p is kept
// only for the lowest common one: item_mask = colOcc(p) below c, kept iff rowOcc(q) & item_mask == 0.
__global__ void __launch_bounds__(256)
k_items(int p0, int np, const int32_t* __restrict__ Acol, const uint16_t* __restrict__ AcolOcc,
        const int64_t* __restrict__ srow_ptr, const int64_t* __restrict__ ioff, int64_t n_items,
        int64_t* __restrict__ plen, int32_t* __restrict__ bfirst, int32_t* __restrict__ item_p,
        uint16_t* __restrict__ item_mask)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) plen[n_items] = 0;
    if (i >= np) return;
    const int p = p0 + i;
    unsigned occ = AcolOcc[p];
    const unsigned all = occ;
    const int64_t* sp = srow_ptr + (size_t)Acol[p] * 16;
    int64_t it = ioff[i];
    while (occ) {
        const int c = __ffs(occ) - 1;
        occ &= occ - 1;
        const int64_t first = sp[c];
        plen[it] = sp[c + 1] - first;
        bfirst[it] = (int32_t)(uint32_t)first;
        item_p[it] = p;
        item_mask[it] = (uint16_t)(all & ((1u << c) - 1u));
        ++it;
    }
}

// widest window over the panel's rows -> scalars[SC_MAXWIN]; total products -> scalars[SC_SUMP]
__global__ void __launch_bounds__(256)
k_max_window(int nrows, const int* __restrict__ jmin, const int* __restrict__ jmax,
             const int64_t* __restrict__ pptr, int np, int64_t* __restrict__ scalars)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    int w = 0;
    if (r < nrows && jmax[r] >= jmin[r]) w = jmax[r] - jmin[r] + 1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) w = max(w, __shfl_xor_sync(0xffffffffu, w, o));
    if ((threadIdx.x & 31) == 0 && w > 0) atomicMax((long long*)&scalars[SC_MAXWIN], (long long)w);
    if (r == 0) scalars[SC_SUMP] = pptr[np];
}

// merge-path split: chunk b starts at diagonal d = b*CHUNK of the (A tile, product) grid; split[b] =
// number of A tiles wholly consumed before it (the chunk's first product is d - split[b])
__global__ void __launch_bounds__(256)
k_merge_split(int nchunks, int np, int64_t P, const int64_t* __restrict__ pptr, int32_t* __restrict__ split)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b > nchunks) return;
    const int64_t d = min((int64_t)b * EX_CHUNK, (int64_t)np + P);
    int64_t lo = max((int64_t)0, d - P), hi = min(d, (int64_t)np);
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (pptr[mid + 1] <= d - mid - 1) lo = mid + 1; else hi = mid;
    }
    split[b] = (int32_t)lo;
}

// Exclusive prefix of this chunk's count over all earlier chunks, found while the kernel runs (decoupled look-back):
// every chunk publishes its own count (AGGREGATE), then walks back over its predecessors' words, 32 at a time,
// summing aggregates until it meets one whose INCLUSIVE prefix is known, and publishes its own inclusive prefix.
// Chunk ids are tickets drawn when a block starts, so every predecessor is already running: no block waits on a
// block that has not been scheduled.  Flag and value share one 64-bit word (single store, no fence needed).
__device__ __forceinline__ int64_t chain_prefix(unsigned long long* state, int b, int64_t mine, int lane)
{
    constexpr unsigned long long AGG = 1ull << 62, INC = 2ull << 62, VAL = (1ull << 62) - 1ull;
    if (lane == 0) atomicExch(&state[b], (b == 0 ? INC : AGG) | (unsigned long long)mine);
    if (b == 0) return 0;
    int64_t prefix = 0;
    for (int j = b - 1;; j -= 32) {
        const int idx = j - lane;
        unsigned long long sv;
        do {
            sv = idx >= 0 ? *reinterpret_cast<volatile unsigned long long*>(&state[idx]) : INC;
        } while (__any_sync(0xffffffffu, (sv >> 62) == 0ull));
        const unsigned inc = __ballot_sync(0xffffffffu, (sv >> 62) == 2ull);
        const int first = inc ? __ffs(inc) - 1 : 31;     // nearest predecessor with a known inclusive prefix
        int64_t v = lane <= first ? (int64_t)(sv & VAL) : 0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        prefix += v;
        if (inc) break;
    }
    if (lane == 0) atomicExch(&state[b], INC | (unsigned long long)(prefix + mine));
    return prefix;
}

// MODE 0: count kept products per chunk.  MODE 1: also write them at out_base[b].  MODE 2: ONE pass: count, find the
// chunk's output offset by look-back over the chunks' counts (chunk_cnt doubles as the look-back state, zeroed by the
// caller; its last entry receives the total) and write the kept products compacted, in product order.
// SLICED: the work items are (A tile, column) pairs over B's row slices (k_items) instead of A tiles
// over B' rows; item_p / srow_tile translate item -> A tile and slice position -> B tile.
template <class KeyT, int MODE, bool SLICED>
__global__ void __launch_bounds__(EX_THREADS, 6)
k_expand(int np, int p0, int rb, int64_t P, const int64_t* __restrict__ pptr, const int32_t* __restrict__ split,
         const int32_t* __restrict__ bfirst, const uint16_t* __restrict__ item_mask,
         const int32_t* __restrict__ item_p, const int32_t* __restrict__ srow_tile,
         const int32_t* __restrict__ Arow, const int32_t* __restrict__ Bcol,
         const uint16_t* __restrict__ BrowOcc, const int* __restrict__ jmin, int wbits, int keep_empty,
         const int64_t* __restrict__ out_base, int64_t* __restrict__ chunk_cnt, int* __restrict__ ticket,
         KeyT* __restrict__ out_key, int2* __restrict__ out_val)
{
    __shared__ int s_rel[EX_CHUNK + 2];       // product offset of slice tile t, relative to the chunk's first product
    __shared__ unsigned s_q0[EX_CHUNK + 1];   // first B tile of tile t's B' row, minus s_rel[t] (mod 2^32)
    __shared__ unsigned short s_occ[EX_CHUNK + 1];
    __shared__ unsigned s_wcnt[EX_WARPS];
    __shared__ int s_chunk;
    __shared__ int64_t s_base;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int chunk = blockIdx.x;
    if (MODE == 2) {                          // chunks in the order the blocks start (see chain_prefix)
        if (tid == 0) s_chunk = atomicAdd(ticket, 1);
        __syncthreads();
        chunk = s_chunk;
    }
    const int64_t total = (int64_t)np + P;
    const int64_t d0 = (int64_t)chunk * EX_CHUNK, d1 = min(d0 + EX_CHUNK, total);
    const int i0 = split[chunk], i1 = split[chunk + 1];
    const int64_t j0 = d0 - i0, j1 = d1 - i1;           // products [j0, j1)
    const int nprod = (int)(j1 - j0);
    const int nt = min(i1 + 1, np) - i0;                // slice tiles [i0, i0 + nt)
    for (int t = tid; t <= nt; t += EX_THREADS) {
        const int64_t rel = pptr[i0 + t] - j0;
        const int r = (int)min(max(rel, (int64_t)INT_MIN), (int64_t)INT_MAX);
        s_rel[t] = r;
        if (t < nt) {
            s_q0[t] = (unsigned)bfirst[i0 + t] - (unsigned)r;
            s_occ[t] = (!SLICED && keep_empty) ? (unsigned short)0xFFFFu : item_mask[i0 + t];
        }
    }
    __syncthreads();
    // lane's products: g = wbase + u*32 + lane (relative to j0)
    const int wbase = warp * (32 * EX_ITEMS);
    int tq[EX_ITEMS];                          // slice tile of item u
    int qq[EX_ITEMS];                          // B tile of item u (-1: none)
    int t = 0;
    {
        const int g = wbase + lane;
        if (g < nprod) {                       // last t in [0, nt) with s_rel[t] <= g
            int lo = 0, hi = nt - 1;
            while (lo < hi) {
                const int mid = (lo + hi + 1) >> 1;
                if (s_rel[mid] <= g) lo = mid; else hi = mid - 1;
            }
            t = lo;
        }
    }
#pragma unroll
    for (int u = 0; u < EX_ITEMS; ++u) {
        const int g = wbase + u * 32 + lane;
        qq[u] = -1;
        tq[u] = 0;
        if (g < nprod) {
            while (s_rel[t + 1] <= g) ++t;     // s_rel[nt] >= nprod ends the walk
            tq[u] = t;
            qq[u] = (int)(s_q0[t] + (unsigned)g);
        }
    }
    if (SLICED) {
#pragma unroll
        for (int u = 0; u < EX_ITEMS; ++u)
            if (qq[u] >= 0) qq[u] = srow_tile[(unsigned)qq[u]];
    }
    unsigned occ[EX_ITEMS];
#pragma unroll
    for (int u = 0; u < EX_ITEMS; ++u) {
        occ[u] = 0u;
        if (qq[u] >= 0 && (!SLICED || s_occ[tq[u]] != 0)) occ[u] = (unsigned)BrowOcc[qq[u]];
    }
    unsigned keepbits = 0, mine = 0;
#pragma unroll
    for (int u = 0; u < EX_ITEMS; ++u) {
        const bool keep = qq[u] >= 0 && (SLICED ? (occ[u] & s_occ[tq[u]]) == 0 : (occ[u] & s_occ[tq[u]]) != 0);
        keepbits |= (unsigned)keep << u;
        mine += keep;
    }
    unsigned wsum = mine;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) wsum += __shfl_xor_sync(0xffffffffu, wsum, o);
    if (lane == 0) s_wcnt[warp] = wsum;
    __syncthreads();
    unsigned before = 0, all = 0;
#pragma unroll
    for (int w = 0; w < EX_WARPS; ++w) {
        const unsigned c = s_wcnt[w];
        before += w < warp ? c : 0u;
        all += c;
    }
    if (MODE != 2 && tid == 0 && chunk_cnt) chunk_cnt[chunk] = all;
    if (MODE == 0) return;
    int64_t pos;
    if (MODE == 2) {
        if (warp == 0) {
            const int64_t prefix = chain_prefix(reinterpret_cast<unsigned long long*>(chunk_cnt), chunk, (int64_t)all, lane);
            if (lane == 0) {
                s_base = prefix;
                if (chunk == (int)gridDim.x - 1) chunk_cnt[gridDim.x] = prefix + (int64_t)all;   // total kept pairs
            }
        }
        __syncthreads();
        pos = s_base + before;
    } else {
        pos = out_base[chunk] + before;
    }
    const unsigned lt = (1u << lane) - 1u;
#pragma unroll
    for (int u = 0; u < EX_ITEMS; ++u) {
        const bool keep = (keepbits >> u) & 1u;
        const unsigned bal = __ballot_sync(0xffffffffu, keep);
        if (keep) {
            const int64_t at = pos + __popc(bal & lt);
            const int p = SLICED ? item_p[i0 + tq[u]] : p0 + i0 + tq[u];
            const int row = Arow[p] - rb;
            const int j = Bcol[qq[u]];
            out_key[at] = ((KeyT)(unsigned)row << wbits) | (KeyT)(unsigned)(j - jmin[row]);
            out_val[at] = make_int2(p, qq[u]);
        }
        pos += __popc(bal);
    }
}

// ---- sort of short rows in shared memory, row by row ---------------------------------------------------
// The compacted pairs are grouped by C' row in row order (products are expanded in A-tile order):
// off[r] = first pair of row r (lower bound of r among the keys' row fields), off[nrows] = F.
template <class KeyT>
__global__ void __launch_bounds__(256)
k_row_offsets(int nrows, const int64_t* __restrict__ d_npairs, int wbits, const KeyT* __restrict__ keys, int* __restrict__ off)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r > nrows) return;
    int lo = 0, hi = (int)*d_npairs;           // the kept-pair count is still on its way to the host
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if ((int64_t)(keys[mid] >> wbits) < (int64_t)r) lo = mid + 1; else hi = mid;
    }
    off[r] = lo;
}

__global__ void __launch_bounds__(256)
k_max_segment(int nrows, const int* __restrict__ off, int64_t* __restrict__ scalars)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    int len = r < nrows ? off[r + 1] - off[r] : 0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) len = max(len, __shfl_xor_sync(0xffffffffu, len, o));
    if ((threadIdx.x & 31) == 0 && len > 0) atomicMax((long long*)&scalars[SC_MAXD], (long long)len);
}

// One warp per C' row, several independent rows per block (no block barrier).  The row's pairs become (tile column,
// position) words in shared memory - position in the low bits makes the words distinct, so the order of equal tile
// columns is the expansion order (ascending A tile), as a stable sort would give.  Rows whose window of tile columns
// fits a small bitmap (stencil / FEM products: a few hundred pairs over a few thousand columns) are ordered WITHOUT a
// comparison network: bitmap of the occupied columns -> popcount prefix = rank of every column = the pair's group
// (its C' tile); a histogram of the groups taken in input order, 32 pairs at a time, gives every pair its rank among
// the earlier pairs of its group (the pairs of one group in a step are __match_any_sync peers, the last of them
// advances the group's count); the scan of the counts gives the group starts, and pair i goes to start(group) + rank.
// The scatter is stable, so every group comes out in position order whatever its size.  Rows with a wider window
// sort the same words with a bitonic network run by the warp.  One pass over the data either way, where the radix
// sort needs one per digit.
constexpr int RS_BMW = 256;            // bitmap words of the counting path: windows of up to 8192 tile columns

// shared memory of one row (one warp) when no row holds more than cap pairs (cap: a power of two >= 32)
constexpr int rs_warp_bytes(int cap) { return cap * 12 + RS_BMW * 6; }

__device__ __forceinline__ unsigned rs_warp_scan(unsigned x, int lane)      // inclusive scan over the warp
{
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned t = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += t;
    }
    return x;
}

template <class KeyT, int POS_BITS>
__global__ void __launch_bounds__(128)
k_row_sort(int nrows, int wbits, int cap, const int* __restrict__ off, const KeyT* __restrict__ in_key,
           const int2* __restrict__ in_val, KeyT* __restrict__ out_key, int2* __restrict__ out_val,
           int64_t* __restrict__ row_tiles)
{
    extern __shared__ __align__(16) unsigned char rs_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int r = blockIdx.x * (blockDim.x >> 5) + warp;
    if (r >= nrows) return;
    const int s = off[r], n = off[r + 1] - s;
    if (n == 0) return;                                  // uniform over the warp
    unsigned* sk = reinterpret_cast<unsigned*>(rs_smem + (size_t)warp * rs_warp_bytes(cap));   // [cap] the row's words
    unsigned* gr = sk + cap;                             // [cap] (group << 16) | rank among the group's earlier pairs
    unsigned* bm = gr + cap;                             // [RS_BMW] occupied tile columns
    unsigned short* cnt = reinterpret_cast<unsigned short*>(bm + RS_BMW);   // [cap] pairs per group -> group starts
    unsigned short* ow = cnt + cap;                      // [cap] positions in output order
    unsigned short* pre = ow + cap;                      // [RS_BMW] distinct columns below each bitmap word
    constexpr int U = 8;                                 // 256 pairs per trip: eight independent global loads in flight
    const KeyT jmask = ((KeyT)1 << wbits) - 1;
    reinterpret_cast<uint4*>(bm)[lane] = make_uint4(0u, 0u, 0u, 0u);
    reinterpret_cast<uint4*>(bm)[lane + 32] = make_uint4(0u, 0u, 0u, 0u);
    __syncwarp();
    unsigned mc = 0;
    for (int b = 0; b < n; b += 32 * U) {
        KeyT k[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int i = b + u * 32 + lane;
            k[u] = i < n ? in_key[s + i] : (KeyT)0;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int i = b + u * 32 + lane;
            if (i < n) {
                const unsigned col = (unsigned)(k[u] & jmask);
                sk[i] = (col << POS_BITS) | (unsigned)i;
                mc = max(mc, col);
                atomicOr(&bm[(col >> 5) & (RS_BMW - 1)], col < (unsigned)RS_BMW * 32u ? 1u << (col & 31) : 0u);
            }
        }
    }
    if (lane < (-n & 31)) sk[n + lane] = 0u;             // pad to whole steps of 32 (cap is a multiple of 32)
    mc = __reduce_max_sync(0xffffffffu, mc);
    __syncwarp();
    const bool counted = mc < (unsigned)RS_BMW * 32u;    // (uniform over the warp)
    unsigned tiles;
    if (counted) {
        {   // the lane's eight bitmap words: distinct columns below each, packed in pairs of 16 bits
            const uint4 a = reinterpret_cast<const uint4*>(bm)[2 * lane], b = reinterpret_cast<const uint4*>(bm)[2 * lane + 1];
            const unsigned c[8] = {(unsigned)__popc(a.x), (unsigned)__popc(a.y), (unsigned)__popc(a.z), (unsigned)__popc(a.w),
                                   (unsigned)__popc(b.x), (unsigned)__popc(b.y), (unsigned)__popc(b.z), (unsigned)__popc(b.w)};
            const unsigned local = c[0] + c[1] + c[2] + c[3] + c[4] + c[5] + c[6] + c[7];
            const unsigned incl = rs_warp_scan(local, lane);
            tiles = __shfl_sync(0xffffffffu, incl, 31);  // the groups ARE the row's C' tiles
            unsigned x = incl - local, p[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                p[q] = x | ((x + c[2 * q]) << 16);
                x += c[2 * q] + c[2 * q + 1];
            }
            reinterpret_cast<uint4*>(pre)[lane] = make_uint4(p[0], p[1], p[2], p[3]);
        }
        for (int g = lane; g < (int)tiles; g += 32) cnt[g] = 0;
        __syncwarp();
        const unsigned lt = (1u << lane) - 1u;
        const int last = ((n + 31) & ~31) - 1;           // last padded word
        for (int b = 0; b < n; b += 32 * U) {            // histogram in input order: rank = earlier pairs of the group
            unsigned g[U];                               // groups of eight steps first: their loads overlap
#pragma unroll
            for (int u = 0; u < U; ++u) g[u] = sk[min(b + u * 32 + lane, last)] >> POS_BITS;
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const unsigned col = g[u];
                g[u] = (pre[col >> 5] + __popc(bm[col >> 5] & ((1u << (col & 31)) - 1u))) | (b + u * 32 + lane < n ? 0u : 0xFFFFu);
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int i = b + u * 32 + lane;
                if (b + u * 32 >= n) break;              // (uniform over the warp)
                const unsigned peers = __match_any_sync(0xffffffffu, g[u]);
                const unsigned rank = cnt[i < n ? g[u] : 0u] + __popc(peers & lt);
                __syncwarp();
                gr[i] = (g[u] << 16) | rank;
                if (i < n && (peers >> lane) == 1u) cnt[g[u]] = (unsigned short)(rank + 1);   // the last peer advances the count
                __syncwarp();
            }
        }
        unsigned carry = 0;                              // group starts: exclusive scan of the counts, 32 groups a step
        for (int g0 = 0; g0 < (int)tiles; g0 += 32) {
            const int g = g0 + lane;
            const unsigned c = g < (int)tiles ? cnt[g] : 0u;
            const unsigned incl = rs_warp_scan(c, lane);
            if (g < (int)tiles) cnt[g] = (unsigned short)(carry + incl - c);
            carry += __shfl_sync(0xffffffffu, incl, 31);
        }
        __syncwarp();
        for (int b = 0; b < n; b += 32 * U) {
            unsigned v[U], d[U];
#pragma unroll
            for (int u = 0; u < U; ++u) v[u] = gr[min(b + u * 32 + lane, last)];
#pragma unroll
            for (int u = 0; u < U; ++u) d[u] = cnt[(v[u] >> 16) & (cap - 1)] + (v[u] & 0xFFFFu);   // (padding: any start, not stored)
#pragma unroll
            for (int u = 0; u < U; ++u)
                if (b + u * 32 + lane < n) ow[d[u]] = (unsigned short)(b + u * 32 + lane);
        }
        __syncwarp();
    } else {                                             // bitonic network over the words
        int N = 2;
        while (N < n) N <<= 1;
        for (int i = n + lane; i < N; i += 32) sk[i] = 0xFFFFFFFFu;
        __syncwarp();
        for (int k = 2; k <= N; k <<= 1)
            for (int j = k >> 1; j > 0; j >>= 1) {
                for (int t = lane; t < (N >> 1); t += 32) {
                    const int lo = ((t & ~(j - 1)) << 1) | (t & (j - 1));      // element with bit j clear
                    const int hi = lo | j;
                    const unsigned a = sk[lo], b = sk[hi];
                    const bool up = (lo & k) == 0;
                    if ((a > b) == up) { sk[lo] = b; sk[hi] = a; }
                }
                __syncwarp();
            }
        unsigned heads = 0;                              // the network does not know the runs of equal tile columns: count them
        for (int i = lane; i < n; i += 32) heads += (i == 0 || (sk[i - 1] >> POS_BITS) != (sk[i] >> POS_BITS)) ? 1u : 0u;
        tiles = __reduce_add_sync(0xffffffffu, heads);
    }
    const KeyT rowbits = (KeyT)(unsigned)r << wbits;
    for (int b = 0; b < n; b += 32 * U) {
        unsigned e[U];
        int2 v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int i = b + u * 32 + lane;
            if (i < n) e[u] = counted ? sk[ow[i]] : sk[i];
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int i = b + u * 32 + lane;
            if (i < n) v[u] = in_val[s + (int)(e[u] & ((1u << POS_BITS) - 1u))];
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int i = b + u * 32 + lane;
            if (i < n) {
                out_key[s + i] = rowbits | (KeyT)(e[u] >> POS_BITS);
                out_val[s + i] = v[u];
            }
        }
    }
    if (lane == 0) row_tiles[r] = (int64_t)tiles;       // C' tiles of this row: scanned into C's row pointer by the caller
}

// C' tiles of the row-sorted pairs: one warp per C' row walks the row's sorted keys, numbers the runs of equal
// tile columns from the row's first tile (row_ptr, the scan of k_row_sort's counts) and writes every tile's
// (row, column, first pair), plus the first tile of every PEM_PAIR_BLOCK-pair block of step 2.  Replaces the
// select of run heads over all pairs + k_ctiles on this path.
template <class KeyT>
__global__ void __launch_bounds__(256)
k_row_tiles(int nrows, int rb, int wbits, int64_t ntiles, int64_t npairs, const int* __restrict__ off,
            const KeyT* __restrict__ keys, const int64_t* __restrict__ row_ptr, const int* __restrict__ jmin,
            int64_t* __restrict__ pair_ptr, int32_t* __restrict__ tile_row, int32_t* __restrict__ tile_col,
            int32_t* __restrict__ pair_blk)
{
    const int row = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (row >= nrows) return;
    if (row == 0 && lane == 0) pair_ptr[ntiles] = npairs;
    const int s = off[row], n = off[row + 1] - s;
    if (n == 0) return;
    const KeyT jmask = ((KeyT)1 << wbits) - 1;
    const int64_t t0 = row_ptr[row];
    const int j0 = jmin[row];
    int running = 0;
    constexpr int U = 8;                                 // 256 pairs per trip: eight independent key loads in flight per lane
    KeyT last = 0;                                       // key of the pair before this trip's first
    for (int base = 0; base < n; base += 32 * U) {
        KeyT k[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int i = base + u * 32 + lane;
            k[u] = i < n ? keys[s + i] : (KeyT)0;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int i = base + u * 32 + lane;
            const bool valid = i < n;
            KeyT kp = __shfl_up_sync(0xffffffffu, k[u], 1);
            if (lane == 0) kp = last;
            last = __shfl_sync(0xffffffffu, k[u], 31);
            const bool head = valid && (i == 0 || kp != k[u]);
            const unsigned bal = __ballot_sync(0xffffffffu, head);
            const int64_t t = t0 + running + __popc(bal & (0xffffffffu >> (31 - lane))) - 1;   // tile of pair s + i
            if (head) {
                pair_ptr[t] = s + i;
                tile_row[t] = rb + row;
                tile_col[t] = j0 + (int)(k[u] & jmask);
            }
            if (valid && ((s + i) & (PEM_PAIR_BLOCK - 1)) == 0) pair_blk[(s + i) / PEM_PAIR_BLOCK] = (int32_t)t;
            running += __popc(bal);
        }
    }
}
constexpr int RS_SMALL = 1024, RS_SMALL_BITS = 10;

template <class KeyT>
struct RunHead {
    const KeyT* keys;
    __device__ __forceinline__ bool operator()(int64_t i) const { return i == 0 || keys[i] != keys[i - 1]; }
};

// thread per C' tile: decode the run's key, open the CSR rows it starts
template <class KeyT>
__global__ void __launch_bounds__(256)
k_ctiles(int64_t ntiles, int64_t npairs, int nrows, int rb, int wbits, const KeyT* __restrict__ keys,
         const int64_t* __restrict__ heads, const int* __restrict__ jmin, int64_t* __restrict__ pair_ptr,
         int32_t* __restrict__ tile_row, int32_t* __restrict__ tile_col, int64_t* __restrict__ row_ptr,
         int32_t* __restrict__ pair_blk)
{
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= ntiles) return;
    const int64_t h = heads[t];
    {   // first tile of every PEM_PAIR_BLOCK-pair block of step 2 (a tile owning pairs [h, hn) opens the blocks that start inside)
        const int64_t hn = t + 1 < ntiles ? heads[t + 1] : npairs;
        for (int64_t b = (h + PEM_PAIR_BLOCK - 1) / PEM_PAIR_BLOCK; b * PEM_PAIR_BLOCK < hn; ++b) pair_blk[b] = (int32_t)t;
    }
    const KeyT key = keys[h];
    const int row = (int)(key >> wbits);
    const int jrel = (int)(key & (((KeyT)1 << wbits) - 1));
    pair_ptr[t] = h;
    tile_row[t] = rb + row;
    tile_col[t] = jmin[row] + jrel;
    const int prev = t ? (int)(keys[heads[t - 1]] >> wbits) : -1;
    for (int r = prev + 1; r <= row; ++r) row_ptr[r] = t;
    if (t == ntiles - 1) {
        for (int r = row + 1; r <= nrows; ++r) row_ptr[r] = ntiles;
        pair_ptr[ntiles] = npairs;
    }
}

__global__ void k_fill_i32(int* p, int n, int v)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

inline int h_bits(int64_t n)
{  // bits needed for values 0..n-1 (at least 1)
    int b = 1;
    while ((int64_t(1) << b) < n) ++b;
    return b;
}

// C's tile arrays, sized for T C' tiles and F pairs (pem_step1_esc left them sized for an empty product)
int alloc_tiles(pem_ctx* ctx, pem_result* C, int64_t T, int64_t F)
{
    if (T >= 0x7fffffffLL)
        return ctx->fail(PEM_ERR_LIMIT, "more than 2^31 C' tiles in one result: multiply in tile-row panels (pem_spgemm_panel)");
    C->tiles = T;
    pem_free(ctx, C->tile_row); pem_free(ctx, C->tile_col); pem_free(ctx, C->pair_ptr);
    PEM_TRY(pem_alloc(ctx, &C->tile_row, (size_t)T));
    PEM_TRY(pem_alloc(ctx, &C->tile_col, (size_t)T));
    PEM_TRY(pem_alloc(ctx, &C->pair_ptr, (size_t)T + 1));
    pem_free(ctx, C->pair_blk);
    return pem_alloc(ctx, &C->pair_blk, (size_t)((F + PEM_PAIR_BLOCK - 1) / PEM_PAIR_BLOCK) + 1);
}

// np work items with product prefix pptr and first-product index bfirst; item_p/srow_tile are null
// for the tile-level expansion (item i = A tile p0 + i) and set for the row-sliced one
template <class KeyT, bool SLICED>
int esc_run(pem_ctx* ctx, const pem_tiled* A, const pem_tiled* B, pem_result* C, int p0, int np, int64_t P,
            int wbits, int rbits, const int64_t* pptr, const int32_t* bfirst, const uint16_t* item_mask,
            const int32_t* item_p, const int* jmin)
{
    const int nrows = C->re - C->rb, rb = C->rb;
    const int64_t total = (int64_t)np + P;
    const int64_t nchunks64 = (total + EX_CHUNK - 1) / EX_CHUNK;
    if (nchunks64 > 0x7ffffff0LL) return ctx->fail(PEM_ERR_LIMIT, "step 1: more than 2^42 tile products");
    const int nchunks = (int)nchunks64;
    Trace tr(ctx->opt_trace != 0);
    tr.mark("esc_run begin");
    int32_t* split = nullptr;
    int64_t* chunk_off = nullptr;
    KeyT *key_a = nullptr, *key_b = nullptr;
    int2 *val_a = nullptr, *val_b = nullptr;
    char* tmp = nullptr;
    int64_t* heads = nullptr;
    int* seg_off = nullptr;
    pem_guard g(ctx, seg_off, split, chunk_off, key_a, key_b, val_a, val_b, tmp, heads);
    PEM_TRY(pem_alloc(ctx, &split, (size_t)nchunks + 1));
    PEM_TRY(pem_alloc(ctx, &chunk_off, (size_t)nchunks + 1));
    k_merge_split<<<pem_div_up((int64_t)nchunks + 1, 256), 256, 0, ctx->stream>>>(nchunks, np, P, pptr, split);
    PEM_LAUNCHED();

    // One expansion into P-sized buffers (the kept count F <= P is not known on the host yet), compacted on the fly.
    // When P-sized buffers would be too large, count first, read F back and write exactly.
    // free device memory, from the context's own books (cudaMemGetInfo takes ~0.7 ms on a B200 box)
    const size_t free_b = ctx->free_at_create > ctx->pool_taken ? ctx->free_at_create - ctx->pool_taken : 0;
    const size_t staged_bytes = (size_t)P * (sizeof(KeyT) + sizeof(int2));
    // (PEM_OPT_ESC_VARIANT bit 0 forces the count-then-write variant; tests use it, nothing else should)
    bool staged = !(ctx->opt_esc_variant & 1) &&
                  staged_bytes <= std::max<size_t>((free_b + ctx->cached_bytes) / 3, (size_t)1 << 28);
    int64_t F = 0, longest_row = 0;
    if (staged && (pem_alloc(ctx, &key_b, (size_t)P) != PEM_OK || pem_alloc(ctx, &val_b, (size_t)P) != PEM_OK)) {
        pem_free(ctx, key_b);              // the books were too optimistic (another process on the GPU?): count first
        pem_free(ctx, val_b);
        staged = false;
    }
    if (staged && (pem_alloc(ctx, &key_a, (size_t)P) != PEM_OK || pem_alloc(ctx, &val_a, (size_t)P) != PEM_OK)) {
        pem_free(ctx, key_a); pem_free(ctx, val_a); pem_free(ctx, key_b); pem_free(ctx, val_b);
        staged = false;
    }
    int* ticket = reinterpret_cast<int*>(ctx->d_scalars + SC_T0);      // zeroed with the other scalars at the start of step 1
    if (staged) {
        // one pass: the chunks' counts are chained by look-back while the kernel runs, the kept pairs land compacted
        PEM_CK(cudaMemsetAsync(chunk_off, 0, ((size_t)nchunks + 1) * 8, ctx->stream));
        PEM_CK(cudaMemsetAsync(ticket, 0, 4, ctx->stream));
        KT_BEGIN(KT_EXPAND);
        k_expand<KeyT, 2, SLICED><<<nchunks, EX_THREADS, 0, ctx->stream>>>(
            np, p0, rb, P, pptr, split, bfirst, item_mask, item_p, B->srow_tile, A->tile_row_idx, B->tile_col_idx,
            B->row_occ, jmin, wbits, ctx->opt_keep_empty, nullptr, chunk_off, ticket, key_a, val_a);
        KT_END(KT_EXPAND);
        PEM_LAUNCHED();
    } else {
        k_expand<KeyT, 0, SLICED><<<nchunks, EX_THREADS, 0, ctx->stream>>>(
            np, p0, rb, P, pptr, split, bfirst, item_mask, item_p, B->srow_tile, A->tile_row_idx, B->tile_col_idx,
            B->row_occ, jmin, wbits, ctx->opt_keep_empty, nullptr, chunk_off, nullptr, nullptr, nullptr);
        PEM_LAUNCHED();
        PEM_CK(cudaMemsetAsync(chunk_off + nchunks, 0, 8, ctx->stream));
        PEM_TRY(pem_scan_exclusive_i64(ctx, chunk_off, (int64_t)nchunks + 1));
    }
    const int64_t* d_F = chunk_off + nchunks;              // kept pairs, on the device
    // Short rows (banded / stencil matrices) are sorted row by row in shared memory: one pass over the
    // pairs.  Power-law inputs have rows of millions of pairs and keep the global radix sort.  Whether every
    // row is short is decided from the longest row, which travels to the host together with F: one stall.
    const bool consider_rows = P < 0x7fffffffLL && wbits + RS_SMALL_BITS <= 32 && !(ctx->opt_esc_variant & 2);
    // every row's segment of the expanded pairs (key_a) and the longest one, into SC_MAXD (left 0 without consider_rows)
    auto row_segments = [&]() -> int {
        PEM_CK(cudaMemsetAsync(ctx->d_scalars + SC_MAXD, 0, 8, ctx->stream));
        if (!consider_rows) return PEM_OK;
        PEM_TRY(pem_alloc(ctx, &seg_off, (size_t)nrows + 1));
        k_row_offsets<KeyT><<<pem_div_up((int64_t)nrows + 1, 256), 256, 0, ctx->stream>>>(nrows, d_F, wbits, key_a, seg_off);
        PEM_LAUNCHED();
        k_max_segment<<<pem_div_up(nrows, 256), 256, 0, ctx->stream>>>(nrows, seg_off, ctx->d_scalars);
        PEM_LAUNCHED();
        return PEM_OK;
    };
    if (staged) {
        PEM_TRY(row_segments());
        {
            pem_size_read rd(ctx);
            int64_t v[2];
            PEM_TRY(rd.add(d_F, 1));
            PEM_TRY(rd.add(ctx->d_scalars + SC_MAXD, 1));
            PEM_TRY(rd.get(v));
            F = v[0];
            longest_row = v[1];
        }
        tr.mark("expand + compact done, F and the longest row known");
        C->pairs = F;
        if (F == 0) return PEM_OK;
    } else {
        {
            pem_size_read rd(ctx);
            PEM_TRY(rd.add(d_F, 1));
            PEM_TRY(rd.get(&F));
        }
        tr.mark("count pass done, F known");
        C->pairs = F;
        if (F == 0) return PEM_OK;
        PEM_TRY(pem_alloc(ctx, &key_a, (size_t)F));
        PEM_TRY(pem_alloc(ctx, &val_a, (size_t)F));
        k_expand<KeyT, 1, SLICED><<<nchunks, EX_THREADS, 0, ctx->stream>>>(
            np, p0, rb, P, pptr, split, bfirst, item_mask, item_p, B->srow_tile, A->tile_row_idx, B->tile_col_idx,
            B->row_occ, jmin, wbits, ctx->opt_keep_empty, chunk_off, nullptr, nullptr, key_a, val_a);
        PEM_LAUNCHED();
        PEM_TRY(pem_alloc(ctx, &key_b, (size_t)F));
        PEM_TRY(pem_alloc(ctx, &val_b, (size_t)F));
        PEM_TRY(row_segments());
        {
            pem_size_read rd(ctx);
            PEM_TRY(rd.add(ctx->d_scalars + SC_MAXD, 1));
            PEM_TRY(rd.get(&longest_row));
        }
    }
    // (a 1024-thread block sorting up to 32768 pairs of a row was tried for config 3's ~13 K-pair rows:
    //  4.5 ms against 2.7 ms for the radix sort)
    const int by_rows = consider_rows && longest_row <= RS_SMALL ? 1 : 0;       // 1: every row holds <= 1024 pairs
    ctx->last_sort_passes = by_rows ? 0 : (wbits + rbits + 7) / 8;
    if (by_rows) {
        KT_BEGIN(KT_SORT);
        int cap = 32;                                   // shared memory by the longest row: short rows keep more warps per SM
        while (cap < longest_row) cap <<= 1;
        const int rows = std::min(4, std::max(1, 32768 / rs_warp_bytes(cap)));     // rows (warps) per block, <= 32 KB
        k_row_sort<KeyT, RS_SMALL_BITS><<<pem_div_up(nrows, rows), 32 * rows, (size_t)rows * rs_warp_bytes(cap), ctx->stream>>>(
            nrows, wbits, cap, seg_off, key_a, val_a, key_b, val_b, C->row_ptr);
        KT_END(KT_SORT);
        PEM_LAUNCHED();
        std::swap(key_a, key_b);
        std::swap(val_a, val_b);
        pem_free(ctx, key_b);
        pem_free(ctx, val_b);
        // the sort counted every row's C' tiles: their scan is C's row pointer, its last entry the tile count
        PEM_TRY(pem_scan_exclusive_i64(ctx, C->row_ptr, (int64_t)nrows + 1));
        int64_t T = 0;
        {
            pem_size_read rd(ctx);
            PEM_TRY(rd.add(C->row_ptr + nrows, 1));
            PEM_TRY(rd.get(&T));
        }
        tr.mark("row sort done, T known");
        PEM_TRY(alloc_tiles(ctx, C, T, F));
        k_row_tiles<KeyT><<<pem_div_up((int64_t)nrows * 32, 256), 256, 0, ctx->stream>>>(
            nrows, rb, wbits, T, F, seg_off, key_a, C->row_ptr, jmin, C->pair_ptr, C->tile_row, C->tile_col, C->pair_blk);
        PEM_LAUNCHED();
        C->pair_list = std::exchange(val_a, nullptr);
        tr.mark("esc_run end (k_row_tiles launched)");
        return PEM_OK;
    } else {   // stable radix sort by (row, column) over the bits in use
        cub::DoubleBuffer<KeyT> dk(key_a, key_b);
        cub::DoubleBuffer<unsigned long long> dv((unsigned long long*)val_a, (unsigned long long*)val_b);
        size_t tb = 0;
        PEM_CK(cub::DeviceRadixSort::SortPairs(nullptr, tb, dk, dv, F, 0, wbits + rbits, ctx->stream));
        PEM_TRY(pem_alloc(ctx, &tmp, tb));
        KT_BEGIN(KT_SORT);
        PEM_CK(cub::DeviceRadixSort::SortPairs(tmp, tb, dk, dv, F, 0, wbits + rbits, ctx->stream));
        KT_END(KT_SORT);
        ctx->launches += 2 + (wbits + rbits + 7) / 8;
        pem_free(ctx, tmp);
        if (dk.Current() != key_a) { std::swap(key_a, key_b); std::swap(val_a, val_b); }
    }
    pem_free(ctx, key_b);
    pem_free(ctx, val_b);
    // heads of the equal-key runs = C' tiles
    int64_t T = 0;
    PEM_TRY(pem_alloc(ctx, &heads, (size_t)F));
    {
        size_t tb = 0;
        thrust::counting_iterator<int64_t> iota(0);
        RunHead<KeyT> pred{key_a};
        int64_t* d_n = ctx->d_scalars + SC_COUNT;
        PEM_CK(cub::DeviceSelect::If(nullptr, tb, iota, heads, d_n, F, pred, ctx->stream));
        PEM_TRY(pem_alloc(ctx, &tmp, tb));
        PEM_CK(cub::DeviceSelect::If(tmp, tb, iota, heads, d_n, F, pred, ctx->stream));
        ctx->launches += 2;
        pem_free(ctx, tmp);
        pem_size_read rd(ctx);
        PEM_TRY(rd.add(d_n, 1));
        PEM_TRY(rd.get(&T));
    }
    tr.mark("sort+select done, T known");
    PEM_TRY(alloc_tiles(ctx, C, T, F));
    k_ctiles<KeyT><<<pem_div_up(T, 256), 256, 0, ctx->stream>>>(T, F, nrows, rb, wbits, key_a, heads, jmin, C->pair_ptr,
                                                                C->tile_row, C->tile_col, C->row_ptr, C->pair_blk);
    PEM_LAUNCHED();
    C->pair_list = std::exchange(val_a, nullptr);
    tr.mark("esc_run end (k_ctiles launched)");
    return PEM_OK;
}

}  // namespace

// called by pem_step1_symbolic (step1.cu) with a fresh result whose row_ptr is allocated
int pem_step1_esc(pem_ctx* ctx, const pem_tiled* A, const pem_tiled* B, pem_result* C)
{
    const int rb = C->rb, re = C->re, nrows = re - rb;
    PEM_CK(cudaMemsetAsync(C->row_ptr, 0, ((size_t)nrows + 1) * 8, ctx->stream));
    PEM_TRY(pem_alloc(ctx, &C->tile_row, 0));
    PEM_TRY(pem_alloc(ctx, &C->tile_col, 0));
    PEM_TRY(pem_alloc(ctx, &C->pair_ptr, 1));
    PEM_CK(cudaMemsetAsync(C->pair_ptr, 0, 8, ctx->stream));
    if (nrows == 0 || A->tiles == 0 || B->tiles == 0) return PEM_OK;
    // A tiles of the panel
    int p0 = 0, p1 = A->tiles;
    if ((rb != 0 || re != A->tile_rows) && A->h_tile_row_ptr.size() == (size_t)A->tile_rows + 1) {
        p0 = A->h_tile_row_ptr[(size_t)rb];      // host copy kept by the conversion: no device read, no sync
        p1 = A->h_tile_row_ptr[(size_t)re];
    } else if (rb != 0 || re != A->tile_rows) {
        int32_t h[2];
        PEM_CK(cudaMemcpyAsync(&h[0], A->tile_row_ptr + rb, 4, cudaMemcpyDeviceToHost, ctx->stream));
        PEM_CK(cudaMemcpyAsync(&h[1], A->tile_row_ptr + re, 4, cudaMemcpyDeviceToHost, ctx->stream));
        PEM_CK(cudaStreamSynchronize(ctx->stream));
        p0 = h[0]; p1 = h[1];
    }
    const int np = p1 - p0;
    if (np == 0) return PEM_OK;
    int64_t *pptr = nullptr, *icnt = nullptr, *pptr_s = nullptr;
    int32_t *bfirst = nullptr, *bfirst_s = nullptr, *item_p = nullptr;
    uint16_t* item_mask = nullptr;
    int *jmin = nullptr, *jmax = nullptr;
    pem_guard g(ctx, pptr, bfirst, jmin, jmax, icnt, pptr_s, bfirst_s, item_p, item_mask);
    // PEM_OPT_STEP1_PATH: 3 forces the tile-level expansion, 4 the row-sliced one; otherwise the
    // cheaper of the two (product counts are known before anything is expanded).  Reference-faithful
    // empty tiles exist only at tile level.
    const bool consider_sliced = !ctx->opt_keep_empty && ctx->opt_step1_path != 3;
    if (consider_sliced) PEM_TRY(pem_tiled_build_srow(ctx, B));
    const int64_t* srow_ptr = consider_sliced ? B->srow_ptr : nullptr;
    PEM_TRY(pem_alloc(ctx, &pptr, (size_t)np + 1));
    PEM_TRY(pem_alloc(ctx, &bfirst, (size_t)np));
    if (consider_sliced) PEM_TRY(pem_alloc(ctx, &icnt, (size_t)np + 1));
    PEM_TRY(pem_alloc(ctx, &jmin, (size_t)nrows));
    PEM_TRY(pem_alloc(ctx, &jmax, (size_t)nrows));
    PEM_CK(cudaMemsetAsync(ctx->d_scalars, 0, PEM_NSCALARS * sizeof(int64_t), ctx->stream));
    k_fill_i32<<<pem_div_up(nrows, 256), 256, 0, ctx->stream>>>(jmin, nrows, INT_MAX);
    PEM_LAUNCHED();
    PEM_CK(cudaMemsetAsync(jmax, 0xFF, (size_t)nrows * 4, ctx->stream));   // -1
    k_tile_products<<<pem_div_up((int64_t)np + 1, 256), 256, 0, ctx->stream>>>(
        p0, np, rb, A->tile_col_idx, A->tile_row_idx, A->col_occ, B->tile_row_ptr, B->tile_col_idx, srow_ptr,
        pptr, bfirst, icnt, jmin, jmax, ctx->d_scalars);
    PEM_LAUNCHED();
    PEM_TRY(pem_scan_exclusive_i64(ctx, pptr, (int64_t)np + 1));
    k_max_window<<<pem_div_up(nrows, 256), 256, 0, ctx->stream>>>(nrows, jmin, jmax, pptr, np, ctx->d_scalars);
    PEM_LAUNCHED();
    int64_t sc[PEM_NSCALARS];
    {
        pem_size_read rd(ctx);                      // stall 1 of a first product (none when a size plan is replayed)
        PEM_TRY(rd.add(ctx->d_scalars + SC_MAXWIN, SC_NLARGE2 - SC_MAXWIN + 1));   // the computed sizes only (not the work-queue cursors)
        PEM_TRY(rd.get(sc + SC_MAXWIN));
    }
    const int64_t P_tile = sc[SC_SUMP];
    const int64_t P_sliced = sc[SC_T2], n_items = sc[SC_T1];
    const int64_t maxw = sc[SC_MAXWIN];
    C->tile_products = P_tile;
    if (P_tile > 0) {
        const int wbits = h_bits(maxw), rbits = h_bits(nrows);
        // the sliced expansion pays an extra indirection per product: take it when it at least halves the products
        const bool sliced = consider_sliced && n_items > 0 && n_items < 0x7fffffffLL && B->srow_total < 0x7fffffffLL &&
                            (ctx->opt_step1_path == 4 || 2 * P_sliced < P_tile);
        if (sliced) {
            C->tile_products = P_sliced;
            PEM_TRY(pem_scan_exclusive_i64(ctx, icnt, (int64_t)np + 1));
            PEM_TRY(pem_alloc(ctx, &pptr_s, (size_t)n_items + 1));
            PEM_TRY(pem_alloc(ctx, &bfirst_s, (size_t)n_items));
            PEM_TRY(pem_alloc(ctx, &item_p, (size_t)n_items));
            PEM_TRY(pem_alloc(ctx, &item_mask, (size_t)n_items));
            k_items<<<pem_div_up(np, 256), 256, 0, ctx->stream>>>(p0, np, A->tile_col_idx, A->col_occ, srow_ptr, icnt, n_items,
                                                                  pptr_s, bfirst_s, item_p, item_mask);
            PEM_LAUNCHED();
            PEM_TRY(pem_scan_exclusive_i64(ctx, pptr_s, n_items + 1));
            if (wbits + rbits <= 32)
                return esc_run<uint32_t, true>(ctx, A, B, C, p0, (int)n_items, P_sliced, wbits, rbits, pptr_s, bfirst_s, item_mask, item_p, jmin);
            else
                return esc_run<uint64_t, true>(ctx, A, B, C, p0, (int)n_items, P_sliced, wbits, rbits, pptr_s, bfirst_s, item_mask, item_p, jmin);
        } else if (wbits + rbits <= 32)
            return esc_run<uint32_t, false>(ctx, A, B, C, p0, np, P_tile, wbits, rbits, pptr, bfirst, A->col_occ + p0, nullptr, jmin);
        else
            return esc_run<uint64_t, false>(ctx, A, B, C, p0, np, P_tile, wbits, rbits, pptr, bfirst, A->col_occ + p0, nullptr, jmin);
    }
    return PEM_OK;
}
