// Step 1: tile-level symbolic SpGEMM  C' = structure(A' * B')  with ordered pair lists.
//
// Replaces, in /root/reference: tile_spgemm_step1_cuda_spa_kernel and ..._numeric_... (spgemm.cu:
// 271-384), the NSPARSE hash path (NSPARSE/spgemm_nsparse_kernel.h, chosen there by the global
// switch `B_tileCols > 512*32`, spgemm.cu:1142) and the CSC-based pair search
// pem_spgemm_step2_search_pairs (spgemm.cu:387-497).  A row-wise expansion that finds a C' tile
// also enumerates the (A tile, B tile) pairs that feed it, so neither the sorted-list
// intersection with its binary searches nor B's tile-level CSC (spgemm.cu:1033-1062) is needed.
//
// Per tile row i of A' (one thread block; 128 threads for ordinary rows, 1024 for heavy ones):
//   window   [jmin, jmax] of tile columns reachable from the row (k_row_window, warp per row)
//   expand   the row's tile products (A tile p) x (B tile q in B' row of p's column) are
//            enumerated FLAT: the A tiles' B'-row extents are staged in shared memory with a
//            prefix sum, product g maps to (p, q) by a shared-memory binary search, and every
//            thread keeps four independent (rowOcc, col) loads in flight.  No thread idles on a
//            short B' row and no warp serialises on a pointer chase.
//   pass A   bitmap of reached tile columns over the window, in shared memory (the SPA of the
//            reference, but windowed, so it costs O(window) not O(B_tileCols) per row); the
//            products that survive the filter below are also written as a compact (p, q, j) list
//   prefix   exclusive popcount scan of the bitmap words: rank(j) = position of tile column j
//            in the ascending C' column list of the row
//   pass B   pairs per C' tile, from the compact list (atomicAdd on counters indexed by rank)
//   scan     -> start of each C' tile's pair list;  emit C' (row, col, pair offset)
//   pass C   place every pair of the compact list at an atomically claimed slot of its list
//   pass D   make every list ascending in k (= ascending A tile id), which is what makes step 3
//            bit-reproducible: short lists are insertion-sorted by one thread, medium ones are
//            rank-sorted by one warp, very long ones (hub tiles) are rebuilt in order by the whole
//            block (binary search of the tile column in each B' row + ordered compaction).  Lists
//            are sets of distinct A tiles, so the final arrays do not depend on the order in
//            which the atomics resolved.
// A pair is dropped (unless PEM_OPT_KEEP_EMPTY_TILES) when colOcc(A tile) & rowOcc(B tile) == 0:
// the 16x16 boolean product of the two tiles is then empty, so C' holds exactly the non-empty
// tiles of C and steps 2/3 never touch a useless pair.
#include <cub/device/device_radix_sort.cuh>

#include <algorithm>
#include <climits>
#include <cstdlib>

#include "engine.cuh"

namespace {

constexpr int TH_SMALL = 128;
constexpr int TH_LARGE = 1024;
constexpr long long LARGE_P = 16384;  // tile products above which a row gets a 1024-thread block
constexpr int LARGE_LA = 512;         // ... or this many A tiles
constexpr int SORT_MAX = 12;          // pair lists up to this length: insertion sort by one thread
constexpr int WSORT_MAX = 256;        // ... up to this length: rank sort by one warp; longer: block rebuild
constexpr int UNROLL = 4;             // independent product loads in flight per thread
// Hash accumulator (the reference's NSPARSE idea, NSPARSE/spgemm_nsparse_kernel.h:464-687, 910-1119): a tile row
// whose products are few but spread over a wide window of tile columns does not clear, scan and popcount a bitmap
// of the whole window; its tile columns go into an open-addressing table in shared memory sized by the row's
// products (linear probing, atomicCAS), the distinct columns are compacted and sorted, and a product finds its
// C' tile by binary search among them.
constexpr int HASH_MAXP = 1024;       // rows with at most this many tile products can take the hash accumulator
constexpr int HASH_SLOTS = 2 * HASH_MAXP;
constexpr int HASH_SPREAD = 16;       // ... automatically when the window holds more than this many columns per product

__device__ __forceinline__ int hash_slots(unsigned P)      // power of two >= 2 * P, at least 64
{
    return max(64, 1 << (33 - __clz(max(P, 1u) - 1u | 1u)));
}
// inserts tile column j; true when it was not in the table yet
__device__ __forceinline__ bool hash_insert(int* tab, int H, int j)
{
    unsigned h = ((unsigned)j * 2654435761u) >> (__clz(H) + 1);
    for (;;) {
        const int old = atomicCAS(&tab[h], -1, j);
        if (old == -1) return true;
        if (old == j) return false;
        h = (h + 1) & (unsigned)(H - 1);
    }
}
// ascending bitonic sort of a[0..n2) (n2 a power of two) by the whole block
template <int THREADS>
__device__ __forceinline__ void block_bitonic(int* a, int n2)
{
    for (int k = 2; k <= n2; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < n2; i += THREADS) {
                const int x = i ^ j;
                if (x > i) {
                    const int u = a[i], v = a[x];
                    if ((u > v) == ((i & k) == 0)) { a[i] = v; a[x] = u; }
                }
            }
            __syncthreads();
        }
}

template <int THREADS>
__device__ __forceinline__ unsigned block_sum(unsigned v, unsigned* red)
{
    constexpr int NW = THREADS / 32;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    unsigned s = 0;
#pragma unroll
    for (int w = 0; w < NW; ++w) s += red[w];
    __syncthreads();
    return s;
}

// In-place exclusive scan of a[0..n) by the whole block; in(i) yields the input of slot i.
template <int THREADS, class In>
__device__ __forceinline__ unsigned block_scan_exclusive(unsigned* a, int n, In in, unsigned* red)
{
    constexpr int NW = THREADS / 32;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int per = (n + THREADS - 1) / THREADS;
    const int b = min(tid * per, n), e = min(b + per, n);
    unsigned local = 0;
    for (int i = b; i < e; ++i) local += in(i);
    unsigned incl = local;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        unsigned t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) red[warp] = incl;
    __syncthreads();
    unsigned woff = 0, total = 0;
#pragma unroll
    for (int w = 0; w < NW; ++w) {
        unsigned x = red[w];
        if (w < warp) woff += x;
        total += x;
    }
    unsigned run = woff + incl - local;
    for (int i = b; i < e; ++i) {
        unsigned x = in(i);
        a[i] = run;
        run += x;
    }
    __syncthreads();
    return total;
}

// Staging area of one chunk of <= THREADS A tiles of the current row.
template <int THREADS>
struct Stage {
    int bs[THREADS];        // first B tile of the A tile's B' row
    unsigned pre[THREADS];  // exclusive prefix of the B' row lengths inside the chunk
    unsigned short occ[THREADS];
};

// Enumerate the kept tile products of A tiles [as, ae): fn(p, q, j) for every B tile q of the B'
// row of A tile p whose boolean product with p is non-empty (or every one if keep_empty).
// Block-wide; all threads must call it.  fn is called with independent loads already resolved.
template <int THREADS, class Fn>
__device__ __forceinline__ void for_each_product(Stage<THREADS>& st, unsigned* red, int as, int ae,
                                                 const int32_t* __restrict__ Acol,
                                                 const uint16_t* __restrict__ AcolOcc,
                                                 const int32_t* __restrict__ Brp,
                                                 const int32_t* __restrict__ Bcol,
                                                 const uint16_t* __restrict__ BrowOcc, int keep_empty, Fn fn)
{
    const int tid = threadIdx.x;
    for (int p0 = as; p0 < ae; p0 += THREADS) {
        const int nch = min(THREADS, ae - p0);
        if (tid < nch) {
            const int k = Acol[p0 + tid];
            const int b = Brp[k];
            st.bs[tid] = b;
            st.occ[tid] = keep_empty ? (unsigned short)0xFFFFu : AcolOcc[p0 + tid];
            st.pre[tid] = (unsigned)(Brp[k + 1] - b);
        }
        __syncthreads();
        const unsigned Pc = block_scan_exclusive<THREADS>(st.pre, nch, [&](int i) { return st.pre[i]; }, red);
        for (unsigned g0 = 0; g0 < Pc; g0 += THREADS * UNROLL) {
            int q[UNROLL], pl[UNROLL];
            unsigned oc[UNROLL];
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) {
                const unsigned g = g0 + u * THREADS + tid;
                q[u] = -1;
                pl[u] = 0;
                oc[u] = 0;
                if (g < Pc) {
                    int lo = 0, hi = nch - 1;            // last c with pre[c] <= g
                    while (lo < hi) {
                        const int mid = (lo + hi + 1) >> 1;
                        if (st.pre[mid] <= g) lo = mid; else hi = mid - 1;
                    }
                    pl[u] = lo;
                    q[u] = st.bs[lo] + (int)(g - st.pre[lo]);
                    oc[u] = st.occ[lo];
                }
            }
            unsigned ro[UNROLL];
            int jj[UNROLL];
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) {
                ro[u] = 0;
                jj[u] = 0;
                if (q[u] >= 0) { ro[u] = BrowOcc[q[u]]; jj[u] = Bcol[q[u]]; }
            }
#pragma unroll
            for (int u = 0; u < UNROLL; ++u)
                if (oc[u] & ro[u]) fn(p0 + pl[u], q[u], jj[u]);
        }
        __syncthreads();
    }
}

// -----------------------------------------------------------------------------------------
// kernel 1: window + tile products per row (warp per tile row) and the row lists for kernel 2
// -----------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_row_window(int rb, int re, const int32_t* __restrict__ Arp, const int32_t* __restrict__ Acol,
             const int32_t* __restrict__ Brp, const int32_t* __restrict__ Bcol,
             int2* __restrict__ win, int32_t* __restrict__ list_small, int32_t* __restrict__ list_large,
             unsigned* __restrict__ key_large, int64_t* __restrict__ scalars, int hash_mode)
{
    int row = rb + (int)((blockIdx.x * (unsigned)blockDim.x + threadIdx.x) >> 5);
    if (row >= re) return;
    int lane = threadIdx.x & 31;
    int jmin = INT_MAX, jmax = -1;
    unsigned long long P = 0;
    const int as = Arp[row], ae = Arp[row + 1];
    for (int p = as + lane; p < ae; p += 32) {
        int k = Acol[p];
        int bs = Brp[k], be = Brp[k + 1];
        if (be > bs) {
            P += (unsigned)(be - bs);
            jmin = min(jmin, Bcol[bs]);
            jmax = max(jmax, Bcol[be - 1]);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        jmin = min(jmin, __shfl_xor_sync(0xffffffffu, jmin, o));
        jmax = max(jmax, __shfl_xor_sync(0xffffffffu, jmax, o));
        P += __shfl_xor_sync(0xffffffffu, P, o);
    }
    if (lane == 0) {
        const long long words = jmax >= 0 ? ((jmax - (jmin & ~31)) >> 5) + 1 : 0;
        const bool heavy = (long long)P > LARGE_P || ae - as > LARGE_LA;
        // accumulator of this row: hash table (hash_mode 1: whenever it fits; 0: when the window is wide for the
        // row's products) or windowed bitmap.  A hash row is marked by a window end below -1 (-jmax - 2).
        const bool hashed = jmax >= 0 && !heavy && P <= (unsigned long long)HASH_MAXP &&
                            (hash_mode == 1 || (hash_mode == 0 && words * 32 > (long long)HASH_SPREAD * (long long)P));
        win[row - rb] = make_int2(jmin, hashed ? -jmax - 2 : jmax);
        if (jmax >= 0) {
            if (hashed) atomicMax((long long*)&scalars[SC_T2], 1ll);
            else atomicMax((long long*)&scalars[SC_MAXWIN], words);
            atomicMax((long long*)&scalars[SC_MAXP], (long long)P);
            atomicAdd((unsigned long long*)&scalars[SC_SUMP], P);
            if (heavy) {
                const unsigned long long at = atomicAdd((unsigned long long*)&scalars[SC_NLARGE1], 1ull);
                list_large[at] = row;
                key_large[at] = ~(unsigned)min(P, 0xFFFFFFFFull);   // ascending sort = heaviest first
            } else
                list_small[atomicAdd((unsigned long long*)&scalars[SC_NSMALL1], 1ull)] = row;
        }
    }
}

// -----------------------------------------------------------------------------------------
// kernel 2 (count): D[row] = C' tiles of the row, F[row] = pairs kept; appends the row to the
// list kernel 3 will take it from (rows whose counters do not fit the small kernel's shared
// memory go to the large one)
// -----------------------------------------------------------------------------------------
template <int THREADS>
__global__ void __launch_bounds__(THREADS)
k_step1_count(const int32_t* __restrict__ rows, int nrows_list, int rb,
              const int32_t* __restrict__ Arp, const int32_t* __restrict__ Acol,
              const uint16_t* __restrict__ AcolOcc, const int32_t* __restrict__ Brp,
              const int32_t* __restrict__ Bcol, const uint16_t* __restrict__ BrowOcc,
              const int2* __restrict__ win, int keep_empty, int dcap_small,
              int64_t* __restrict__ D, int64_t* __restrict__ F,
              int32_t* __restrict__ list_small, int32_t* __restrict__ list_large,
              unsigned* __restrict__ key_large, int64_t* __restrict__ scalars,
              unsigned long long* __restrict__ work)
{
    extern __shared__ unsigned sm[];
    __shared__ unsigned red[THREADS / 32 + 1];
    __shared__ Stage<THREADS> st;
    __shared__ int s_li;
    const int tid = threadIdx.x;
    for (;;) {                                      // rows are handed out through a work queue
        if (tid == 0) s_li = (int)atomicAdd(work, 1ull);
        __syncthreads();
        const int li = s_li;
        __syncthreads();
        if (li >= nrows_list) break;
        const int row = rows[li];
        const int2 wnd = win[row - rb];
        unsigned f = 0, d = 0;
        if (wnd.y < -1) {                           // hash accumulator: distinct tile columns counted at insertion
            int* tab = reinterpret_cast<int*>(sm);
            const int as = Arp[row], ae = Arp[row + 1];
            unsigned P = 0;
            for (int p = as + tid; p < ae; p += THREADS) {
                const int k = Acol[p];
                P += (unsigned)(Brp[k + 1] - Brp[k]);
            }
            P = block_sum<THREADS>(P, red);
            const int H = hash_slots(P);
            for (int w = tid; w < H; w += THREADS) tab[w] = -1;
            __syncthreads();
            for_each_product<THREADS>(st, red, as, ae, Acol, AcolOcc, Brp, Bcol, BrowOcc, keep_empty,
                                      [&](int, int, int j) {
                                          d += hash_insert(tab, H, j) ? 1u : 0u;
                                          ++f;
                                      });
        } else {
            const int base = wnd.x & ~31;
            const int W = ((wnd.y - base) >> 5) + 1;
            for (int w = tid; w < W; w += THREADS) sm[w] = 0;
            __syncthreads();
            for_each_product<THREADS>(st, red, Arp[row], Arp[row + 1], Acol, AcolOcc, Brp, Bcol, BrowOcc, keep_empty,
                                      [&](int, int, int j) {
                                          j -= base;
                                          atomicOr(&sm[j >> 5], 1u << (j & 31));
                                          ++f;
                                      });
            for (int w = tid; w < W; w += THREADS) d += __popc(sm[w]);
        }
        d = block_sum<THREADS>(d, red);
        f = block_sum<THREADS>(f, red);
        if (tid == 0 && d > 0) {
            D[row - rb] = d;
            F[row - rb] = f;
            atomicMax((long long*)&scalars[SC_MAXD], (long long)d);
            if (THREADS == TH_LARGE || (int)d > dcap_small) {
                const unsigned long long at = atomicAdd((unsigned long long*)&scalars[SC_NLARGE2], 1ull);
                list_large[at] = row;
                key_large[at] = ~f;                                 // ascending sort = most pairs first
            } else
                list_small[atomicAdd((unsigned long long*)&scalars[SC_NSMALL2], 1ull)] = row;
        }
    }
}

// -----------------------------------------------------------------------------------------
// kernel 3 (fill).  Shared memory: bitmap[Wmax] | prefix[Wmax] | cnt[dcap]; rows with more than
// dcap C' tiles keep cnt in this block's slice of a global scratch.  tmp_p/tmp_q/tmp_j hold the
// compact list of kept products of every row at the row's pair offset.
// -----------------------------------------------------------------------------------------
template <int THREADS>
__global__ void __launch_bounds__(THREADS)
k_step1_fill(const int32_t* __restrict__ rows, int nrows_list, int rb,
             const int32_t* __restrict__ Arp, const int32_t* __restrict__ Acol,
             const uint16_t* __restrict__ AcolOcc, const int32_t* __restrict__ Brp,
             const int32_t* __restrict__ Bcol, const uint16_t* __restrict__ BrowOcc,
             const int2* __restrict__ win, int keep_empty, int Wmax, int dcap,
             unsigned* __restrict__ gscratch, size_t gstride,
             int2* __restrict__ tmp_pq, int32_t* __restrict__ tmp_j,
             const int64_t* __restrict__ c_row_ptr, const int64_t* __restrict__ pair_row_ptr,
             int32_t* __restrict__ c_tile_row, int32_t* __restrict__ c_tile_col,
             int64_t* __restrict__ pair_ptr, int2* __restrict__ pairs,
             unsigned long long* __restrict__ work, unsigned long long* __restrict__ prof)
{
    extern __shared__ unsigned sm[];
    constexpr int NW = THREADS / 32;
    __shared__ unsigned red[NW + 1];
    __shared__ unsigned longmask[NW];
    __shared__ unsigned wsortmask[NW];
    __shared__ unsigned cursor;
    // the staging area is only live during pass A, the warp-sort slabs only during pass D
    __shared__ union { Stage<THREADS> st; int wslab[NW * WSORT_MAX]; } u;
    unsigned* bitmap = sm;
    unsigned* prefix = sm + Wmax;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    long long tprev = prof ? clock64() : 0;
    const long long tstart = tprev;
    __shared__ int s_li;
#define PROF_MARK(i) do { if (prof && tid == 0) { long long t_ = clock64(); atomicAdd(&prof[i], (unsigned long long)(t_ - tprev)); tprev = t_; } } while (0)
    for (;;) {                                      // rows are handed out through a work queue
        if (tid == 0) s_li = (int)atomicAdd(work, 1ull);
        __syncthreads();
        const int li = s_li;
        __syncthreads();
        if (li >= nrows_list) break;
        const int row = rows[li];
        const int64_t cbase = c_row_ptr[row - rb];
        const int D = (int)(c_row_ptr[row - rb + 1] - cbase);
        const int64_t pbase = pair_row_ptr[row - rb];
        const int F = (int)(pair_row_ptr[row - rb + 1] - pbase);
        const int2 wnd = win[row - rb];
        const bool hashed = wnd.y < -1;             // hash accumulator: table in the bitmap's place, sorted columns behind it
        const int base = hashed ? 0 : wnd.x & ~31;
        const int W = hashed ? 0 : ((wnd.y - base) >> 5) + 1;
        int* tab = reinterpret_cast<int*>(sm);
        int* cols = tab;                            // hash rows: set below (behind the table)
        int H = 0;
        unsigned* cnt = (D <= dcap) ? sm + 2 * (size_t)Wmax : gscratch + (size_t)blockIdx.x * gstride;
        if (hashed) {
            H = hash_slots((unsigned)F);            // F kept products <= the row's products: 2 * F slots hold them
            cols = tab + H;
            for (int w = tid; w < H; w += THREADS) tab[w] = -1;
        }
        for (int w = tid; w < W; w += THREADS) bitmap[w] = 0;
        for (int i = tid; i < D; i += THREADS) cnt[i] = 0;
        if (tid == 0) cursor = 0;
        __syncthreads();
        const int as = Arp[row], ae = Arp[row + 1];
        // pass A: reached tile columns + compact list of the kept products
        int2* tpq = tmp_pq + pbase;
        int32_t* tj = tmp_j + pbase;
        int2* prow = pairs + pbase;
        for_each_product<THREADS>(u.st, red, as, ae, Acol, AcolOcc, Brp, Bcol, BrowOcc, keep_empty,
                                  [&](int p, int q, int j) {
                                      j -= base;
                                      if (hashed) hash_insert(tab, H, j);
                                      else atomicOr(&bitmap[j >> 5], 1u << (j & 31));
                                      // warp-aggregated slot claim
                                      const unsigned act = __activemask();
                                      const int leader = __ffs(act) - 1;
                                      unsigned slot = 0;
                                      if (lane == leader) slot = atomicAdd(&cursor, (unsigned)__popc(act));
                                      slot = __shfl_sync(act, slot, leader) + __popc(act & ((1u << lane) - 1u));
                                      tpq[slot] = make_int2(p, q); tj[slot] = j;
                                  });
        PROF_MARK(0);
        if (hashed) {
            // the table's D distinct columns, compacted behind it and sorted ascending (padded to a power of two)
            int D2 = 1;
            while (D2 < D) D2 <<= 1;
            if (tid == 0) cursor = 0;
            __syncthreads();
            for (int w = tid; w < H; w += THREADS) {
                const int j = tab[w];
                if (j >= 0) cols[atomicAdd(&cursor, 1u)] = j;
            }
            for (int i = D + tid; i < D2; i += THREADS) cols[i] = INT_MAX;
            __syncthreads();
            block_bitonic<THREADS>(cols, D2);
        } else
            block_scan_exclusive<THREADS>(prefix, W, [&](int i) { return (unsigned)__popc(bitmap[i]); }, red);
        PROF_MARK(1);
        // pass B: pairs per C' tile; the list's j is replaced by its rank
        for (int i = tid; i < F; i += THREADS) {
            const int j = tj[i];
            unsigned rank;
            if (hashed) {                           // position of j among the sorted columns
                int lo = 0, hi = D - 1;
                while (lo < hi) {
                    const int mid = (lo + hi) >> 1;
                    if (cols[mid] < j) lo = mid + 1; else hi = mid;
                }
                rank = (unsigned)lo;
            } else {
                const int w = j >> 5;
                rank = prefix[w] + __popc(bitmap[w] & ((1u << (j & 31)) - 1u));
            }
            tj[i] = (int)rank;
            atomicAdd(&cnt[rank], 1u);
        }
        __syncthreads();
        PROF_MARK(2);
        block_scan_exclusive<THREADS>(cnt, D, [&](int i) { return cnt[i]; }, red);
        PROF_MARK(3);
        // emit the C' tiles of this row (columns ascending) with their pair offsets
        if (hashed)
            for (int r = tid; r < D; r += THREADS) {
                c_tile_row[cbase + r] = row;
                c_tile_col[cbase + r] = cols[r];
                pair_ptr[cbase + r] = pbase + cnt[r];
            }
        for (int w = tid; w < W; w += THREADS) {
            unsigned m = bitmap[w];
            unsigned r = prefix[w];
            while (m) {
                int b = __ffs(m) - 1;
                m &= m - 1;
                c_tile_row[cbase + r] = row;
                c_tile_col[cbase + r] = base + w * 32 + b;
                pair_ptr[cbase + r] = pbase + cnt[r];
                ++r;
            }
        }
        __syncthreads();
        PROF_MARK(4);
        // pass C: placement (slot claimed atomically; cnt[r] ends as the END of list r)
        for (int i = tid; i < F; i += THREADS) {
            const unsigned pos = atomicAdd(&cnt[tj[i]], 1u);
            prow[pos] = tpq[i];
        }
        __syncthreads();
        PROF_MARK(5);
        // pass D: ascending k inside every list
        for (int r0 = 0; r0 < D; r0 += THREADS) {
            const int r = r0 + tid;
            int cls = 0;                               // 1: warp rank sort, 2: block rebuild
            if (r < D) {
                const unsigned s = r ? cnt[r - 1] : 0u, e = cnt[r];
                const unsigned len = e - s;
                if (len > (unsigned)WSORT_MAX) {
                    cls = 2;
                } else if (len > (unsigned)SORT_MAX) {
                    cls = 1;
                } else if (len >= 2) {
                    int2* pl = prow + s;
                    for (unsigned i = 1; i < len; ++i) {
                        const int2 key = pl[i];
                        int jx = (int)i - 1;
                        while (jx >= 0 && pl[jx].x > key.x) {
                            pl[jx + 1] = pl[jx];
                            --jx;
                        }
                        pl[jx + 1] = key;
                    }
                }
            }
            const unsigned balw = __ballot_sync(0xffffffffu, cls == 1);
            const unsigned ball = __ballot_sync(0xffffffffu, cls == 2);
            if (lane == 0) { wsortmask[warp] = balw; longmask[warp] = ball; }
            __syncthreads();
            // medium lists: one warp each, rank sort on the A tile ids staged in shared memory
            {
                int turn = 0;
                for (int w = 0; w < NW; ++w) {
                    unsigned m = wsortmask[w];
                    while (m) {
                        const int rr = r0 + w * 32 + __ffs(m) - 1;
                        m &= m - 1;
                        if ((turn++ % NW) != warp) continue;
                        const unsigned s = rr ? cnt[rr - 1] : 0u;
                        const int n = (int)(cnt[rr] - s);
                        int2* pl = prow + s;
                        int* slab = u.wslab + warp * WSORT_MAX;
                        int ma[WSORT_MAX / 32], mb[WSORT_MAX / 32];
#pragma unroll
                        for (int i = 0; i < WSORT_MAX / 32; ++i) {
                            const int x = i * 32 + lane;
                            const int2 v = x < n ? pl[x] : make_int2(INT_MAX, 0);
                            ma[i] = v.x;
                            mb[i] = v.y;
                            if (x < n) slab[x] = ma[i];
                        }
                        __syncwarp();
                        int rk[WSORT_MAX / 32];
#pragma unroll
                        for (int i = 0; i < WSORT_MAX / 32; ++i) rk[i] = 0;
                        for (int x = 0; x < n; ++x) {
                            const int v = slab[x];
#pragma unroll
                            for (int i = 0; i < WSORT_MAX / 32; ++i) rk[i] += (v < ma[i]);
                        }
#pragma unroll
                        for (int i = 0; i < WSORT_MAX / 32; ++i)
                            if (i * 32 + lane < n) pl[rk[i]] = make_int2(ma[i], mb[i]);
                        __syncwarp();
                    }
                }
            }
            // very long lists (hub tiles): rebuilt in order by the whole block
            for (int w = 0; w < NW; ++w) {
                unsigned m = longmask[w];
                while (m) {                                    // block-uniform loop
                    const int rr = r0 + w * 32 + __ffs(m) - 1;
                    m &= m - 1;
                    const int jr = c_tile_col[cbase + rr];
                    unsigned outp = rr ? cnt[rr - 1] : 0u;
                    for (int p0 = as; p0 < ae; p0 += THREADS) {
                        const int p = p0 + tid;
                        int q = -1;
                        if (p < ae) {
                            const int k = Acol[p];
                            int lo = Brp[k], hi = Brp[k + 1] - 1;
                            while (lo <= hi) {
                                int mid = (lo + hi) >> 1;
                                int v = Bcol[mid];
                                if (v == jr) { q = mid; break; }
                                if (v < jr) lo = mid + 1; else hi = mid - 1;
                            }
                            if (q >= 0 && !keep_empty && !(AcolOcc[p] & BrowOcc[q])) q = -1;
                        }
                        const unsigned hit = __ballot_sync(0xffffffffu, q >= 0);
                        if (lane == 0) red[warp] = __popc(hit);
                        __syncthreads();
                        unsigned before = 0, total = 0;
#pragma unroll
                        for (int x = 0; x < NW; ++x) {
                            unsigned c = red[x];
                            if (x < warp) before += c;
                            total += c;
                        }
                        if (q >= 0) {
                            const unsigned pos = outp + before + __popc(hit & ((1u << lane) - 1u));
                            prow[pos] = make_int2(p, q);
                        }
                        outp += total;
                        __syncthreads();
                    }
                }
            }
            __syncthreads();
        }
        PROF_MARK(6);
    }
    if (prof && tid == 0) atomicMax(&prof[7], (unsigned long long)(clock64() - tstart));
#undef PROF_MARK
}

__global__ void k_set_i64(int64_t* p, int64_t idx, int64_t v) { p[idx] = v; }

}  // namespace

extern "C" int pem_step1_symbolic(pem_ctx* ctx, const pem_tiled* A, const pem_tiled* B,
                                  int32_t rb, int32_t re, pem_result** out)
{
    PEM_RANGE("pem_step1_symbolic");
    if (!out) return PEM_ERR_ARG;
    *out = nullptr;
    if (!ctx || !A || !B) return PEM_ERR_ARG;
    if (A->cols != B->rows) return ctx->fail(PEM_ERR_ARG, "inner dimensions differ (A.cols != B.rows)");
    if (A->dtype != B->dtype) return ctx->fail(PEM_ERR_ARG, "operands have different value types");
    if (rb < 0 || re < rb || re > A->tile_rows) return ctx->fail(PEM_ERR_ARG, "tile-row panel out of range");
    PEM_CK(cudaSetDevice(ctx->device));
    auto result_free = [ctx](pem_result* r) { pem_result_free(ctx, r); };
    std::unique_ptr<pem_result, decltype(result_free)> C(new pem_result(), result_free);
    C->dtype = A->dtype;
    C->a_uid = A->uid; C->b_uid = B->uid;
    C->keep_empty = ctx->opt_keep_empty != 0;
    C->rb = rb; C->re = re; C->rows = A->rows; C->cols = B->cols; C->tile_cols = B->tile_cols;
    const int nrows = re - rb;
    ctx->last_sort_passes = -1;
    // small operands are launch-bound: the per-row bitmap path below needs ~8 launches and 2 host
    // syncs, expand-sort-compress ~20 and 3
    const bool small = (int64_t)A->tiles + B->tiles <= 65536 && B->tile_cols <= 65536;
    if ((ctx->opt_step1_path >= 2 && ctx->opt_step1_path != 5) || (ctx->opt_step1_path == 0 && !small)) {     // expand-sort-compress (step1_esc.cu)
        PEM_TRY(pem_alloc(ctx, &C->row_ptr, (size_t)nrows + 1));
        PEM_TRY(pem_step1_esc(ctx, A, B, C.get()));
        C->stage = 1;
        *out = C.release();
        return PEM_OK;
    }
    int64_t* pair_row_ptr = nullptr;
    int2* win = nullptr;
    int32_t *l1s = nullptr, *l1l = nullptr, *l2s = nullptr, *l2l = nullptr, *lsorted = nullptr;
    unsigned *key_l = nullptr, *key_sorted = nullptr;
    char* sort_tmp = nullptr;
    int2* tmp_pq = nullptr;
    int32_t* tmp_j = nullptr;
    unsigned* gscr = nullptr;
    unsigned long long* prof = nullptr;
    pem_guard g(ctx, pair_row_ptr, win, l1s, l1l, l2s, l2l, gscr, prof, lsorted, key_l, key_sorted, sort_tmp, tmp_pq, tmp_j);
    PEM_TRY(pem_alloc(ctx, &C->row_ptr, (size_t)nrows + 1));
    PEM_TRY(pem_alloc(ctx, &pair_row_ptr, (size_t)nrows + 1));
    PEM_TRY(pem_alloc(ctx, &win, (size_t)nrows));
    PEM_TRY(pem_alloc(ctx, &l1s, (size_t)nrows)); PEM_TRY(pem_alloc(ctx, &l1l, (size_t)nrows));
    PEM_TRY(pem_alloc(ctx, &l2s, (size_t)nrows)); PEM_TRY(pem_alloc(ctx, &l2l, (size_t)nrows));
    PEM_TRY(pem_alloc(ctx, &lsorted, (size_t)nrows));
    PEM_TRY(pem_alloc(ctx, &key_l, (size_t)nrows)); PEM_TRY(pem_alloc(ctx, &key_sorted, (size_t)nrows));
    size_t sort_bytes = 0;
    PEM_CK(cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, key_l, key_sorted, l1l, lsorted, nrows > 0 ? nrows : 1, 0, 32, ctx->stream));
    PEM_TRY(pem_alloc(ctx, &sort_tmp, sort_bytes));
    unsigned long long* work = (unsigned long long*)(ctx->d_scalars + SC_WORK0);
    // heavy rows are taken from the work queue heaviest first (longest-processing-time order)
    auto sort_heavy = [&](int32_t*& list, int64_t n) -> int {
        if (n < 2) return PEM_OK;
        size_t b = sort_bytes;
        PEM_CK(cub::DeviceRadixSort::SortPairs(sort_tmp, b, key_l, key_sorted, list, lsorted, (int)n, 0, 32, ctx->stream));
        ctx->launches += 3;
        std::swap(list, lsorted);
        return PEM_OK;
    };
    PEM_CK(cudaMemsetAsync(ctx->d_scalars, 0, PEM_NSCALARS * sizeof(int64_t), ctx->stream));
    PEM_CK(cudaMemsetAsync(C->row_ptr, 0, ((size_t)nrows + 1) * 8, ctx->stream));
    PEM_CK(cudaMemsetAsync(pair_row_ptr, 0, ((size_t)nrows + 1) * 8, ctx->stream));

    const bool any = nrows > 0 && A->tiles > 0 && B->tiles > 0;
    int64_t maxwin = 0, maxd = 0, n1s = 0, n1l = 0, n2s = 0, n2l = 0;
    if (any) {
        // PEM_OPT_STEP1_PATH 5: hash accumulators wherever a row's products fit the table; 1 / automatic: only for rows
        // whose window is wide for their products
        k_row_window<<<pem_div_up((int64_t)nrows * 32, 256), 256, 0, ctx->stream>>>(
            rb, re, A->tile_row_ptr, A->tile_col_idx, B->tile_row_ptr, B->tile_col_idx, win, l1s, l1l, key_l, ctx->d_scalars,
            ctx->opt_step1_path == 5 ? 1 : 0);
        PEM_LAUNCHED();
        int64_t sc[PEM_NSCALARS];
        pem_size_read rd(ctx);
        PEM_TRY(rd.add(ctx->d_scalars + SC_MAXWIN, SC_NLARGE2 - SC_MAXWIN + 1));   // the computed sizes only (not the work-queue cursors)
        PEM_TRY(rd.get(sc + SC_MAXWIN));
        maxwin = sc[SC_MAXWIN];
        if (sc[SC_T2]) maxwin = std::max<int64_t>(maxwin, HASH_SLOTS);     // hash rows: table (and sorted columns) in the bitmap's place
        C->tile_products = sc[SC_SUMP];
        n1s = sc[SC_NSMALL1]; n1l = sc[SC_NLARGE1];
    }
    // shared-memory plan (dynamic part; the kernels also hold the staging area / sort slabs and a
    // few words statically, which count against the same 227 KB)
    const size_t win_bytes = (size_t)maxwin * 4;
    const size_t static_small = std::max<size_t>((size_t)(TH_SMALL / 32) * WSORT_MAX * 4, (size_t)TH_SMALL * 12) + 1024;
    const size_t static_large = std::max<size_t>((size_t)(TH_LARGE / 32) * WSORT_MAX * 4, (size_t)TH_LARGE * 12) + 1024;
    const size_t budget = (size_t)ctx->smem_optin;
    const int dcap_small = 2048;
    const size_t smem_fill_small = 2 * win_bytes + (size_t)dcap_small * 4;
    if (maxwin > 0 && (smem_fill_small + static_small > budget || 2 * win_bytes + static_large + 32768 > budget))
        return ctx->fail(PEM_ERR_LIMIT, "step 1: a tile row's column window exceeds the shared-memory bitmap "
                                        "(more than ~600K tile columns within one tile row's reach)");
    // counters of the heavy-row kernel: at most what fits, but only half the SM when 8K counters
    // still fit in that half, so that two heavy-row blocks stay resident per SM
    size_t dl = (budget - 2 * win_bytes - static_large) / 4;
    if (budget / 2 > 2 * win_bytes + static_large + 8192 * 4) dl = (budget / 2 - 2 * win_bytes - static_large) / 4;
    const int dcap_large = (int)dl;
    const size_t smem_fill_large = 2 * win_bytes + (size_t)dcap_large * 4;
    if (n1s + n1l > 0) {
        PEM_CK(cudaFuncSetAttribute(k_step1_count<TH_SMALL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)win_bytes));
        PEM_CK(cudaFuncSetAttribute(k_step1_count<TH_LARGE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)win_bytes));
        PEM_TRY(sort_heavy(l1l, n1l));
        if (n1l > 0) {  // heavy rows first: they are the tail
            int grid = (int)std::min<int64_t>(n1l, (int64_t)ctx->sm_count * 2);
            k_step1_count<TH_LARGE><<<grid, TH_LARGE, win_bytes, ctx->stream>>>(
                l1l, (int)n1l, rb, A->tile_row_ptr, A->tile_col_idx, A->col_occ, B->tile_row_ptr, B->tile_col_idx,
                B->row_occ, win, ctx->opt_keep_empty, dcap_small, C->row_ptr, pair_row_ptr, l2s, l2l, key_l, ctx->d_scalars, work + 0);
            PEM_LAUNCHED();
        }
        if (n1s > 0) {
            int grid = (int)std::min<int64_t>(n1s, (int64_t)ctx->sm_count * 16);
            k_step1_count<TH_SMALL><<<grid, TH_SMALL, win_bytes, ctx->stream>>>(
                l1s, (int)n1s, rb, A->tile_row_ptr, A->tile_col_idx, A->col_occ, B->tile_row_ptr, B->tile_col_idx,
                B->row_occ, win, ctx->opt_keep_empty, dcap_small, C->row_ptr, pair_row_ptr, l2s, l2l, key_l, ctx->d_scalars, work + 1);
            PEM_LAUNCHED();
        }
        PEM_TRY(pem_scan_exclusive_i64(ctx, C->row_ptr, (int64_t)nrows + 1));
        PEM_TRY(pem_scan_exclusive_i64(ctx, pair_row_ptr, (int64_t)nrows + 1));
        PEM_CK(cudaMemcpyAsync(&ctx->d_scalars[SC_T0], C->row_ptr + nrows, 8, cudaMemcpyDeviceToDevice, ctx->stream));
        PEM_CK(cudaMemcpyAsync(&ctx->d_scalars[SC_T1], pair_row_ptr + nrows, 8, cudaMemcpyDeviceToDevice, ctx->stream));
        int64_t sc[PEM_NSCALARS];
        pem_size_read rd(ctx);
        PEM_TRY(rd.add(ctx->d_scalars + SC_MAXWIN, SC_NLARGE2 - SC_MAXWIN + 1));   // the computed sizes only (not the work-queue cursors)
        PEM_TRY(rd.get(sc + SC_MAXWIN));
        C->tiles = sc[SC_T0];
        C->pairs = sc[SC_T1];
        maxd = sc[SC_MAXD];
        n2s = sc[SC_NSMALL2]; n2l = sc[SC_NLARGE2];
    }
    PEM_TRY(pem_alloc(ctx, &C->tile_row, (size_t)C->tiles));
    PEM_TRY(pem_alloc(ctx, &C->tile_col, (size_t)C->tiles));
    PEM_TRY(pem_alloc(ctx, &C->pair_ptr, (size_t)C->tiles + 1));
    PEM_TRY(pem_alloc(ctx, &C->pair_list, (size_t)C->pairs));
    if (C->pairs > 0) {
        PEM_TRY(pem_alloc(ctx, &tmp_pq, (size_t)C->pairs));
        PEM_TRY(pem_alloc(ctx, &tmp_j, (size_t)C->pairs));
    }
    const bool want_prof = ctx->opt_trace > 1;      // PEM_OPT_TRACE = 2: per-phase cycle counters of the bitmap kernels
    if (want_prof) {
        PEM_TRY(pem_alloc(ctx, &prof, 16));
        PEM_CK(cudaMemsetAsync(prof, 0, 16 * 8, ctx->stream));
    }
    auto report = [&](const char* which, int grid) -> int {
        unsigned long long h[8];
        PEM_CK(cudaMemcpyAsync(h, prof, sizeof h, cudaMemcpyDeviceToHost, ctx->stream));
        PEM_CK(cudaStreamSynchronize(ctx->stream));
        fprintf(stderr, "[step1 %s: cycles summed over %d blocks] passA %llu scanW %llu passB %llu scanD %llu emit %llu "
                        "passC %llu passD %llu | slowest block %llu cycles\n", which, grid, h[0], h[1], h[2], h[3], h[4], h[5], h[6], h[7]);
        PEM_CK(cudaMemsetAsync(prof, 0, 16 * 8, ctx->stream));
        return PEM_OK;
    };
    PEM_TRY(sort_heavy(l2l, n2l));
    if (n2l > 0) {
        const bool two_per_sm = 2 * (smem_fill_large + static_large) <= budget;
        int grid = (int)std::min<int64_t>(n2l, (int64_t)ctx->sm_count * (two_per_sm ? 2 : 1));
        size_t stride = 0;
        if (maxd > dcap_large) {
            stride = (size_t)maxd;
            PEM_TRY(pem_alloc(ctx, &gscr, stride * (size_t)grid));
        }
        PEM_CK(cudaFuncSetAttribute(k_step1_fill<TH_LARGE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_fill_large));
        k_step1_fill<TH_LARGE><<<grid, TH_LARGE, smem_fill_large, ctx->stream>>>(
            l2l, (int)n2l, rb, A->tile_row_ptr, A->tile_col_idx, A->col_occ, B->tile_row_ptr, B->tile_col_idx, B->row_occ,
            win, ctx->opt_keep_empty, (int)maxwin, dcap_large, gscr, stride, tmp_pq, tmp_j, C->row_ptr, pair_row_ptr,
            C->tile_row, C->tile_col, C->pair_ptr, C->pair_list, work + 2, prof);
        PEM_LAUNCHED();
        if (want_prof) PEM_TRY(report("fill<1024>", grid));
    }
    if (n2s > 0) {
        int grid = (int)std::min<int64_t>(n2s, (int64_t)ctx->sm_count * 16);
        PEM_CK(cudaFuncSetAttribute(k_step1_fill<TH_SMALL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_fill_small));
        k_step1_fill<TH_SMALL><<<grid, TH_SMALL, smem_fill_small, ctx->stream>>>(
            l2s, (int)n2s, rb, A->tile_row_ptr, A->tile_col_idx, A->col_occ, B->tile_row_ptr, B->tile_col_idx, B->row_occ,
            win, ctx->opt_keep_empty, (int)maxwin, dcap_small, nullptr, 0, tmp_pq, tmp_j, C->row_ptr, pair_row_ptr,
            C->tile_row, C->tile_col, C->pair_ptr, C->pair_list, work + 3, prof);
        PEM_LAUNCHED();
        if (want_prof) PEM_TRY(report("fill<128>", grid));
    }
    k_set_i64<<<1, 1, 0, ctx->stream>>>(C->pair_ptr, C->tiles, C->pairs);
    PEM_LAUNCHED();
    C->stage = 1;
    *out = C.release();
    return PEM_OK;
}
