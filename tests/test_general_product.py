"""General A*B products: independently built rectangular operands, inputs constructed at the kernels' selection
thresholds (each at n and n+1, with the observable that tells which side ran), and IEEE special values compared
bit for bit, including the sign of zero.

Every other parity test multiplies A*A or A*A^T, where A.tile_rows == B.tile_cols and both operands have the same
density; here m, k and n differ, and A and B are hypersparse (one or two nonzeros per tile) or dense (at least eight)
independently of each other.

The constructed inputs put a chosen number of (A tile, B tile) pairs into a C' tile: A tile (I, K) for K = 0..p-1
with a nonzero in local column 0, B tile (K, J) with a nonzero in local row 0.  C' tile (I, J) then has exactly p
pairs; the number of such J is the length of the C' row, the span of the J its window.  A B tile whose nonzeros sit
only in local row 1 makes a pair that is reachable but empty (kept only with PEM_OPT_KEEP_EMPTY_TILES).

Observables: ``last_sort_passes`` is -1 when step 1 took the per-row path, 0 when expand-sort-compress sorted row by
row in shared memory, otherwise the radix passes (wbits + rbits + 7) // 8 of the global sort (4 for 32-bit keys at
32 key bits, 5 for 64-bit keys at 33); ``info.tile_products`` tells the row-sliced expansion from the tile-level one;
``last_step3_kernel`` is 1 row-owner, 2 entry-owner, 3 tile-class, 4 window kernel."""
import math

import numpy as np
import pytest
import scipy.sparse as sp

import pem_spgemm_b200 as pem
from oracle import host, tiles

gpu = pytest.mark.gpu
PATHS = (0, 1, 3, 4, 5)          # PEM_OPT_STEP1_PATH: automatic, bitmap, tile-level ESC, row-sliced ESC, hash rows


def _assert_bits(v, vo, tag=""):
    """Bit equality of two value arrays: the sign of zero counts, and a NaN matches any NaN (payloads
    legitimately differ between the host and the GPU).  np.array_equal would take -0.0 for +0.0 and fail on NaN."""
    v, vo = np.asarray(v), np.asarray(vo)
    assert v.dtype == vo.dtype and v.shape == vo.shape, (tag, v.dtype, vo.dtype, v.shape, vo.shape)
    u = np.uint32 if v.dtype == np.float32 else np.uint64
    if np.array_equal(v.view(u), vo.view(u)):
        return
    nan, nano = np.isnan(v), np.isnan(vo)
    assert np.array_equal(nan, nano), f"{tag} NaN at {np.flatnonzero(nan != nano)[:10]}"
    bad = np.flatnonzero((v.view(u) != vo.view(u)) & ~nan)
    assert bad.size == 0, f"{tag} {bad.size} values differ in their bits, first at {bad[:10]}: {v[bad[:5]]} vs {vo[bad[:5]]}"


# ---------------------------------------------------------------------------------------------------------------
# input generators
# ---------------------------------------------------------------------------------------------------------------
class Mat:
    """A sparse matrix under construction, entry by entry (explicit zeros, -0.0, Inf and NaN are kept)."""

    def __init__(self, rows, cols):
        self.rows, self.cols, self.e = rows, cols, {}

    def put(self, i, j, v):
        assert 0 <= i < self.rows and 0 <= j < self.cols, (i, j, self.rows, self.cols)
        self.e[(int(i), int(j))] = v

    def tile(self, I, J, r, c, v):
        self.put(16 * I + r, 16 * J + c, v)

    def coo(self):
        keys = sorted(self.e)
        I = np.array([k[0] for k in keys], np.int32)
        J = np.array([k[1] for k in keys], np.int32)
        V = np.array([self.e[k] for k in keys], np.float64)
        return self.rows, self.cols, I, J, V


def _rand_tiled(rows, cols, ntiles, per_tile, rng):
    """ntiles distinct random tiles of a rows x cols matrix, each with per_tile = (lo, hi) nonzeros (fewer only
    where a ragged edge tile has fewer positions), values uniform(-1, 1)."""
    tr, tc = -(-rows // 16), -(-cols // 16)
    I, J = [], []
    for t in rng.choice(tr * tc, size=min(ntiles, tr * tc), replace=False):
        ti, tj = divmod(int(t), tc)
        h, w = min(16, rows - 16 * ti), min(16, cols - 16 * tj)
        k = min(h * w, int(rng.integers(per_tile[0], per_tile[1] + 1)))
        loc = rng.choice(h * w, size=k, replace=False)
        I.append(16 * ti + loc // w); J.append(16 * tj + loc % w)
    I = np.concatenate(I).astype(np.int32); J = np.concatenate(J).astype(np.int32)
    o = np.lexsort((J, I))
    return rows, cols, I[o], J[o], rng.uniform(-1, 1, I.size)


class Fmt:
    """Constants of one value type for the special-value witnesses."""

    def __init__(self, dt):
        self.dt = dt
        fi = np.finfo(dt)
        self.eps_half = float(fi.epsneg)                       # 2^-53 / 2^-24: half an ulp of 1
        self.big = 2.0 ** (fi.maxexp - 1)                      # 2^1023 / 2^127
        self.tiny = float(fi.smallest_subnormal)               # 2^-1074 / 2^-149
        self.sub_max = float(fi.smallest_normal) - self.tiny   # largest subnormal
        e = fi.minexp                                          # -1022 / -126
        self.neg_small = -(2.0 ** (e // 2))                    # a normal A value whose products with `under` (normal
        self.under = 2.0 ** (e // 2 - 60)                      # too) are below half the smallest subnormal


F64, F32 = Fmt(np.float64), Fmt(np.float32)


def pair_family(p, shift=0, dense=False, fmt=F64, rng=None):
    """One tile row of C': tile (0, 0) with `shift` pairs (random values), then tile (0, 1) with exactly p pairs,
    K = 0..p-1 in ascending order.  Tile (0, 1) carries the witnesses: A(0, 16K) = 1, so C(0, 16 + c) is the sum of
    B(16K, 16 + c) over K in ascending order:
      c0: [1, h, h, 0, ...]          h = half an ulp of 1: 1 in order, 1 + 2h if the two small products come first
      c1: [0, ..., 1, h, h]          the same at the end of the list
      c2: [big, big, -big, 0, ...]   big = 2^1023: Inf in order, big if reordered
      c3: [0, ..., big, big, -big]
      c4: smallest / largest subnormal alternating
      c5: `under` everywhere: row 1 (A = neg_small) underflows to -0.0 from the first fma on
      c6: Inf at the last pair: Inf in row 0, -Inf in row 1, NaN in row 2 (A = +0.0 opposite the Inf)
      c7: NaN at the first pair, -1 elsewhere: NaN in rows 0, 1 and 3, +0.0 in row 2
      c8: -tiny at the first pair, 0 elsewhere: -tiny in row 0, +0.0 in rows 1 and 3
    Row 3 has one A entry, -0.0 at K = 0: every product of it is an exact zero, so its entries are +0.0 (a sum
    started from -0.0 would give -0.0).  ``dense`` adds 64 random nonzeros to every A tile (rows 4-11, columns 1-8)
    and 104 to every B tile (rows 1-8), which makes both operands dense without touching the witness rows."""
    rng = rng or np.random.default_rng(p * 1000 + shift)
    nk = max(p, shift, 1)
    A = Mat(13, 16 * nk - 3)
    B = Mat(16 * nk - 3, 29)
    f = fmt
    for K in range(nk):
        A.tile(0, K, 0, 0, 1.0)
        if dense:
            for r in range(4, 12):
                for c in range(1, 9):
                    A.tile(0, K, r, c, float(fmt.dt(rng.uniform(-1, 1))))
    for K in range(shift):
        B.tile(K, 0, 0, 0, float(fmt.dt(rng.uniform(-1, 1))))
        B.tile(K, 0, 0, 3, float(fmt.dt(rng.uniform(-1, 1))))
    for K in range(p):
        A.tile(0, K, 1, 0, f.neg_small)
        col = [0.0] * 9
        col[0] = 1.0 if K == 0 else f.eps_half if K in (1, 2) else 0.0
        col[1] = 1.0 if K == p - 3 else f.eps_half if K in (p - 2, p - 1) else 0.0
        col[2] = f.big if K in (0, 1) else -f.big if K == 2 else 0.0
        col[3] = f.big if K in (p - 3, p - 2) else -f.big if K == p - 1 else 0.0
        col[4] = f.tiny if K % 2 == 0 else f.sub_max
        col[5] = f.under
        col[6] = math.inf if K == p - 1 else 1.0
        col[7] = math.nan if K == 0 else -1.0
        col[8] = -f.tiny if K == 0 else 0.0
        for c, v in enumerate(col):
            B.tile(K, 1, 0, c, v)
    A.tile(0, p - 1, 2, 0, 0.0)
    A.tile(0, 0, 3, 0, -0.0)
    if dense:
        for K in range(nk):
            for J in range(2):
                if (J == 1 and K < p) or (J == 0 and K < shift):
                    for r in range(1, 9):
                        for c in range(13):
                            B.tile(K, J, r, c, float(fmt.dt(rng.uniform(-1, 1))))
    return A, B


def window_case(width, tile_rows=1):
    """A (16 * tile_rows - 7 rows) times B whose tile row 0 has tiles at tile columns 0 and width - 1: every C' row
    reaching B's tile row 0 has a window of exactly `width` tile columns.  A's last tile row has one entry too."""
    A = Mat(16 * tile_rows - 7, 13)
    B = Mat(13, 16 * (width - 1) + 5)
    for I in range(tile_rows):
        A.tile(I, 0, 0, 0, 1.5 + I)
    A.tile(tile_rows - 1, 0, 8, 4, -0.75)
    B.tile(0, 0, 0, 0, 2.0); B.tile(0, 0, 4, 2, 0.5)
    B.tile(0, width - 1, 0, 1, -3.0); B.tile(0, width - 1, 4, 4, 0.25)
    return A, B


def empty_span_case(n_empty):
    """keep-empty: C' tile row 0 = tile 0 (16 entries), n_empty reachable empty tiles (their B tiles hold nonzeros
    in local row 1 only, A's tiles only in local column 0), then a tile of 208 entries.  The first 128-entry block
    of the entry-owner kernel then spans n_empty + 2 C' tiles."""
    A = Mat(16, 29)
    B = Mat(29, 16 * (n_empty + 2) - 3)
    for r in range(16):
        A.tile(0, 0, r, 0, 1.0 + r)
        A.tile(0, 1, r, 0, 0.5 - r)
    B.tile(0, 0, 0, 0, 3.0)
    for J in range(1, n_empty + 1):
        B.tile(0, J, 1, J % 13, 7.0)
    for c in range(13):
        B.tile(1, n_empty + 1, 0, c, 0.125 * (c + 1))
    return A, B


def step2_form_case(a_short, b_short):
    """Three pairs into one C tile of 8 entries (8 < 4 * 3, so the automatic step 3 choice follows the hit words).
    Every A and B tile holds 8 nonzeros (dense by the step-2 rule A.nnz >= 8 * A.tiles), except one tile of the
    operand marked short, which holds 7."""
    A = Mat(16, 45)
    B = Mat(45, 16)
    for K in range(3):
        for r in range(8 - (1 if a_short and K == 1 else 0)):
            A.tile(0, K, r, 0, 1.0 + r + K)
        B.tile(K, 0, 0, 0, 0.5 + K)
        for r in range(1, 8 - (1 if b_short and K == 2 else 0)):
            B.tile(K, 0, r, 5, -1.0 - r)
    return A, B


def entries_per_pair_case(nnz):
    """One pair, one C tile of `nnz` entries (step 3 takes the window kernel at nnz >= 4 * pairs)."""
    A = Mat(5, 9)
    B = Mat(9, 21)
    A.put(0, 0, 1.25)
    for c in range(nnz):
        B.put(0, c, 0.5 + c)
    return A, B


def heavy_row_case(P):
    """Tile row 0 of A with 64 tiles, each reaching 256 B tiles: 16384 tile products, or 16385 with one more B tile
    (LARGE_P).  Tile row 1 is a light companion: one A tile reaching B's tile row 0 (256 products)."""
    A = Mat(32, 16 * 64)
    B = Mat(16 * 64, 16 * 257)
    rng = np.random.default_rng(P)
    for K in range(64):
        A.tile(0, K, 0, 0, float(rng.uniform(-1, 1)))
        for J in range(256):
            B.tile(K, J, 0, J % 16, float(rng.uniform(-1, 1)))
    for x in range(P - 64 * 256):
        B.tile(x, 256, 0, 0, 1.0)
    A.tile(1, 0, 3, 0, 0.5)
    return A, B


def many_a_tiles_case(na):
    """Tile row 0 of A with na tiles, each reaching one B tile: na A tiles and na tile products (LARGE_LA at 512).
    Tile row 1 is a light companion: one A tile reaching one B tile."""
    A = Mat(32, 16 * na)
    B = Mat(16 * na, 16 * 8)
    rng = np.random.default_rng(na)
    for K in range(na):
        A.tile(0, K, 0, 0, float(rng.uniform(-1, 1)))
        B.tile(K, K % 8, 0, K % 16, float(rng.uniform(-1, 1)))
    A.tile(1, 0, 5, 0, -1.5)
    return A, B


def hash_row_case(P, width):
    """Tile row 0 of A with 4 tiles (far from LARGE_LA), each reaching 256 B tiles spread over `width` tile columns:
    1024 tile products, or 1025 with one more B tile (HASH_MAXP).  The window is wide for the products (more than
    16 tile columns per product), so the automatic choice hashes the row whenever it may."""
    A = Mat(16, 16 * 4 - 5)
    B = Mat(16 * 4 - 5, 16 * (width - 1) + 7)
    rng = np.random.default_rng(P + width)
    Js = np.linspace(0, width - 1, 256).round().astype(np.int64)
    assert np.unique(Js).size == 256 and 1 not in Js
    for K in range(4):
        A.tile(0, K, K, 0, float(rng.uniform(-1, 1)))
        for J in Js:
            B.tile(K, int(J), 0, int(J + K) % 7, float(rng.uniform(-1, 1)))
    for _ in range(P - 1024):
        B.tile(0, 1, 0, 3, 2.0)
    return A, B


def spread_case(jmax):
    """Tile row 0 of A with 4 tiles, each reaching 16 B tiles whose tile columns span 0..jmax: 64 tile products over
    a window of (jmax >> 5) + 1 bitmap words.  The automatic choice hashes the row when words * 32 > 16 * 64
    (HASH_SPREAD), i.e. from jmax = 1024 on."""
    A = Mat(16, 16 * 4 - 5)
    B = Mat(16 * 4 - 5, 16 * jmax + 9)
    rng = np.random.default_rng(jmax)
    Js = np.linspace(0, jmax, 16).round().astype(np.int64)
    for K in range(4):
        A.tile(0, K, 2 * K, 0, float(rng.uniform(-1, 1)))
        for J in Js:
            B.tile(K, int(J), 0, int(J) % 9, float(rng.uniform(-1, 1)))
    return A, B


def _row_stats(A, B):
    """Per tile row of A: (A tiles, tile products, bitmap words of the tile-column window), as the per-row path's
    first kernel computes them (step1.cu, k_row_window)."""
    TA, TB = tiles.tile_format(*A.coo()), tiles.tile_format(*B.coo())
    out = []
    for I in range(TA.tile_rows):
        ks = TA.tile_col[TA.tile_row_ptr[I]:TA.tile_row_ptr[I + 1]]
        P, jmin, jmax = 0, 1 << 40, -1
        for k in ks:
            bs, be = int(TB.tile_row_ptr[k]), int(TB.tile_row_ptr[k + 1])
            if be > bs:
                P += be - bs
                jmin, jmax = min(jmin, int(TB.tile_col[bs])), max(jmax, int(TB.tile_col[be - 1]))
        out.append((int(ks.size), P, ((jmax - (jmin & ~31)) >> 5) + 1 if jmax >= 0 else 0))
    return out


def diag_tiles_case(na, nb):
    """A with na diagonal tiles times B with nb tiles (diagonal, plus tile (0, 1) when nb > na)."""
    n = 16 * na
    A = Mat(n, n)
    B = Mat(n, n)
    for t in range(na):
        A.tile(t, t, 0, 0, 1.0 + t % 7)
        B.tile(t, t, 0, 1, 0.5 - t % 5)
    for t in range(nb - na):
        B.tile(0, t + 1, 0, 2, 3.0)
    return A, B


def _csr(M):
    return host.coo_to_csr(*M.coo())


def _oracle(A, B, f32=False):
    oA, oB = _csr(A), _csr(B)
    threads = int(host.lib().oracle_max_threads())
    if B.cols > 1 << 22:                    # the oracle's accumulator is B.cols wide in every thread
        host.set_threads(2)
    try:
        return oA, oB, (host.spgemm_f32 if f32 else host.spgemm)(oA, oB)
    finally:
        host.set_threads(threads)


def _is_dense(M):
    T = tiles.tile_format(*M.coo())
    return T.vals.size >= 8 * T.cnt


def _tile_product(A, B, keep):
    return tiles.tiled_product(tiles.tile_format(*A.coo()), tiles.tile_format(*B.coo()), keep_empty=keep)


# ---------------------------------------------------------------------------------------------------------------
# CPU: the generators do what they claim, and the oracle against an implementation that shares none of its code
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("p,shift", [(12, 0), (13, 31), (145, 127), (1025, 0), (1025, 127)])
def test_pair_family_has_the_claimed_pairs(p, shift):
    A, B = pair_family(p, shift, dense=True)
    for keep in (False, True):
        P = _tile_product(A, B, keep)
        assert list(P.c_tile_col) == ([0, 1] if shift else [1])
        assert list(np.diff(P.pair_ptr)) == ([shift, p] if shift else [p])
        assert list(P.c_row_ptr) == [0, P.c_tile_col.size]
        ta = P.pairs_a[P.pair_ptr[-2]:]
        assert np.all(np.diff(ta) > 0)                  # ascending k
    TA, TB = tiles.tile_format(*A.coo()), tiles.tile_format(*B.coo())
    assert TA.vals.size >= 8 * TA.cnt and TB.vals.size >= 8 * TB.cnt


@pytest.mark.parametrize("width,tile_rows", [(8192, 1), (8193, 1), (1 << 22, 1), ((1 << 22) + 1, 1),
                                             ((1 << 22) + 1, 512), ((1 << 22) + 1, 513)])
def test_window_case_has_the_claimed_window(width, tile_rows):
    A, B = window_case(width, tile_rows)
    TA, TB = tiles.tile_format(*A.coo()), tiles.tile_format(*B.coo())
    assert TA.tile_rows == tile_rows and TB.tile_cols == width
    P = tiles.tiled_product(TA, TB, keep_empty=True)
    assert P.c_tile_col.size == 2 * tile_rows
    for I in range(tile_rows):
        cols = P.c_tile_col[P.c_row_ptr[I]:P.c_row_ptr[I + 1]]
        assert cols.max() - cols.min() + 1 == width


@pytest.mark.parametrize("n_empty", [510, 511])
def test_empty_span_case_has_the_claimed_tiles(n_empty):
    A, B = empty_span_case(n_empty)
    P = _tile_product(A, B, True)
    nnz = np.diff(P.c_tile_nnz_ptr)
    assert nnz.size == n_empty + 2 and nnz[0] == 16 and nnz[-1] == 208 and not nnz[1:-1].any()
    assert _tile_product(A, B, False).c_tile_col.size == 2


def test_small_cases_have_the_claimed_counts():
    for a_short, b_short in ((0, 0), (1, 0), (0, 1)):
        A, B = step2_form_case(a_short, b_short)
        TA, TB = tiles.tile_format(*A.coo()), tiles.tile_format(*B.coo())
        assert (TA.vals.size >= 8 * TA.cnt) == (not a_short) and (TB.vals.size >= 8 * TB.cnt) == (not b_short)
        P = tiles.tiled_product(TA, TB, keep_empty=False)
        assert P.pairs_a.size == 3 and P.c_tile_nnz_ptr[-1] == 8
    for nb in (32768, 32769):
        A, B = diag_tiles_case(32768, nb)
        assert tiles.tile_format(*A.coo()).cnt + tiles.tile_format(*B.coo()).cnt == 32768 + nb


def test_per_row_cases_straddle_their_thresholds():
    """The per-row path's rules, restated on the constructed inputs: a row is heavy above LARGE_P = 16384 tile
    products or LARGE_LA = 512 A tiles; it may take the hash table up to HASH_MAXP = 1024 products when not heavy,
    automatically when words * 32 > HASH_SPREAD (16) * products."""
    for x in (16384, 16385):
        (la, P, _), light = _row_stats(*heavy_row_case(x))
        assert (la, P) == (64, x) and light[0] <= 512 and light[1] <= 16384
    for x in (512, 513):
        (la, P, _), light = _row_stats(*many_a_tiles_case(x))
        assert (la, P) == (x, x) and P <= 16384 and light[0] <= 512 and light[1] <= 16384
    for x in (1024, 1025):
        for width in (20000, 1 << 20):
            [(la, P, words)] = _row_stats(*hash_row_case(x, width))
            assert (la, P) == (4, x) and words * 32 > 16 * P
            assert words == (width - 1) // 32 + 1 and (width <= 65536) == (words <= 2048)
    for jmax, hashed in ((1023, False), (1024, True)):
        [(la, P, words)] = _row_stats(*spread_case(jmax))
        assert (la, P) == (4, 64) and (words * 32 > 16 * P) == hashed


def _dyadic(rows, cols, nnz, seed):
    """Random entries k * 2^e with |k| <= 7 and -4 <= e <= 4: every product and every partial sum of the
    products below is exact in fp64, so any summation order gives the same bits."""
    rng = np.random.default_rng(seed)
    key = np.unique(rng.integers(0, rows * cols, nnz))
    k = rng.integers(-7, 8, key.size); k[k == 0] = 1
    V = k * np.exp2(rng.integers(-4, 5, key.size)).astype(np.float64)
    return rows, cols, (key // cols).astype(np.int32), (key % cols).astype(np.int32), V


@pytest.mark.parametrize("m,k,n,seed", [(37, 530, 9011, 1), (4003, 203, 37, 2), (300, 17, 301, 3), (1, 1000, 1, 4),
                                        (129, 61, 2, 5)])
def test_oracle_general_product_vs_scipy_exact(m, k, n, seed):
    """host.spgemm(A, B) on independent rectangular operands: structure against scipy on all-ones patterns
    (scipy drops exact zeros), values against scipy exactly (dyadic values), cancelled entries +0.0."""
    a = _dyadic(m, k, max(1, m * k // 7), seed)
    b = _dyadic(k, n, max(1, k * n // 9), seed + 100)
    oA, oB = host.coo_to_csr(*a), host.coo_to_csr(*b)
    oC = host.spgemm(oA, oB)
    assert (oC.rows, oC.cols) == (m, n)
    pa = sp.csr_matrix((np.ones(a[2].size), (a[2], a[3])), shape=(m, k))
    pb = sp.csr_matrix((np.ones(b[2].size), (b[2], b[3])), shape=(k, n))
    R = (pa @ pb).tocsr(); R.sort_indices()
    assert np.array_equal(oC.ptr, R.indptr.astype(np.int64)) and np.array_equal(oC.idx, R.indices.astype(np.int32))
    assert host.flop(oA, oB) == int(R.sum())
    D = (sp.csr_matrix((a[4], (a[2], a[3])), shape=(m, k)) @ sp.csr_matrix((b[4], (b[2], b[3])), shape=(k, n))).toarray()
    r, c, v = oC.to_coo()
    want = D[r, c] + 0.0                                    # scipy's cancelled sums: +0.0
    _assert_bits(v, want)
    assert not np.any((v == 0) & np.signbit(v))            # exact cancellation gives +0.0, never -0.0
    if v.size > 10000:
        assert np.count_nonzero(v == 0) > 0                 # large products do cancel somewhere


@pytest.mark.parametrize("fmt", ["f64", "f32"])
@pytest.mark.parametrize("p", [12, 1025])
def test_oracle_special_value_witnesses(fmt, p):
    """The oracle's semantics on the witnesses of pair_family, against hand-derived bits."""
    f = F64 if fmt == "f64" else F32
    A, B = pair_family(p, 0, fmt=f)
    oA, oB, oC = _oracle(A, B, f32=fmt == "f32")
    dt = f.dt
    r, c, v = oC.to_coo()
    got = {(int(i), int(j) - 16): x for i, j, x in zip(r, c, v)}
    one = dt(1.0)
    bits = lambda x: np.array([x], dt).view(np.uint32 if dt == np.float32 else np.uint64)[0]
    assert bits(got[(0, 0)]) == bits(one) and bits(got[(0, 1)]) == bits(one)          # ascending k
    assert got[(0, 2)] == np.inf and got[(0, 3)] == np.inf                               # overflow kept
    assert got[(0, 4)] != 0 and abs(got[(0, 4)]) < np.finfo(dt).smallest_normal * p     # subnormals survive
    assert got[(1, 5)] == 0 and np.signbit(got[(1, 5)])                                  # fma underflow: -0.0
    assert got[(0, 6)] == np.inf and got[(1, 6)] == -np.inf and np.isnan(got[(2, 6)])    # 0 * Inf = NaN
    assert np.isnan(got[(0, 7)]) and np.isnan(got[(1, 7)]) and np.isnan(got[(3, 7)])
    assert got[(2, 7)] == 0 and not np.signbit(got[(2, 7)])
    assert bits(got[(0, 8)]) == bits(dt(-f.tiny)) and not np.signbit(got[(1, 8)])
    for j in (0, 1, 2, 3, 4, 5, 6, 8):                                                    # exact zeros from +0.0
        assert got[(3, j)] == 0 and not np.signbit(got[(3, j)]), j
    isnan = np.isnan(v)
    assert {(int(i), int(j) - 16) for i, j in zip(r[isnan], c[isnan])} == {(2, 6), (0, 7), (1, 7), (3, 7)}


# ---------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------
class Opts:
    """Engine options for the duration of a block, restored to their defaults afterwards."""
    DEFAULTS = {pem.OPT_STEP1_PATH: 0, pem.OPT_STEP2_KERNEL: 0, pem.OPT_OWNER: 0, pem.OPT_KEEP_EMPTY_TILES: 0}

    def __init__(self, engine, **kw):
        self.engine = engine
        self.kw = {getattr(pem, "OPT_" + k.upper()): v for k, v in kw.items()}

    def __enter__(self):
        for o, v in self.kw.items():
            self.engine.set_option(o, v)

    def __exit__(self, *a):
        for o in self.kw:
            self.engine.set_option(o, self.DEFAULTS.get(o, 0))


def _expected_s3(owner, step2, a_dense, b_dense, nnz, pairs):
    """The step-3 kernel the engine picks (spgemm.cu step 2 / step3.cu pem_step3_numeric)."""
    if owner == 1:
        return 1
    if owner == 3:
        return 3
    rows_form = step2 == 3 or (step2 == 0 and a_dense)
    hits = not (step2 == 0 and rows_form and owner in (0, 4) and b_dense)
    return 4 if owner == 4 or not hits or (owner == 0 and nnz >= 4 * pairs) else 2


def _dense(T):
    return T.info.nnz >= 8 * T.info.tiles


def _convert(engine, M, f32=False):
    return engine.convert_coo(*M.coo(), dtype=np.float32 if f32 else np.float64)


def _product(engine, tA, tB, nparts=1):
    """C = A*B in nparts tile-row panels: (rows, cols, vals) concatenated, and the infos of the panels."""
    bounds = engine.partition_panels(tA, tB, nparts)
    assert bounds[0] == 0 and bounds[-1] == tA.info.tile_rows
    parts, infos = [], []
    for q in range(nparts):
        C = engine.spgemm(tA, tB, panel=(bounds[q], bounds[q + 1]))
        parts.append(C.to_coo()); infos.append(C.info)
        C.free()
    return [np.concatenate([x[j] for x in parts]) for j in range(3)], infos


def _assert_same(got, oC, tag=""):
    r, c, v = got
    ro, co, vo = oC.to_coo()
    assert np.array_equal(r, ro) and np.array_equal(c, co), tag
    assert np.array_equal(np.isinf(v), np.isinf(vo)) and np.array_equal(np.isnan(v), np.isnan(vo)), tag
    _assert_bits(v, vo, tag)


SHAPES = {"wide": (37, 1203, 9011, 150, 3000), "tall": (4003, 1203, 37, 3000, 150)}    # m, k, n, A tiles, B tiles
DENSITY = {"hyper": (1, 2), "dense": (9, 16)}


@gpu
@pytest.mark.parametrize("shape", ["wide", "tall"])
@pytest.mark.parametrize("da,db", [("hyper", "hyper"), ("hyper", "dense"), ("dense", "hyper"), ("dense", "dense")])
def test_general_product_every_variant(engine, shape, da, db):
    """Independent A (m x k) and B (k x n), every step-1 path x step-2 kernel x step-3 owner: C' structure, pair lists,
    masks and tile offsets against the tile oracle, values bit for bit against the host oracle, C's shape, the flop
    count, the CSR export and the step-3 kernel that ran.  Keep-empty and the panel count are a fractional design, not
    a full cross product: each (path, step-2, owner) triple runs with one keep-empty setting, (path + step2 + owner) % 2,
    and in three panels when (step2 + owner) % 3 == 0, else in one; over the 100 triples both keep-empty settings and
    both panel counts meet every path, step-2 kernel and owner."""
    m, k, n, ta, tb = SHAPES[shape]
    rng = np.random.default_rng(sum(map(ord, shape + da + db)))
    a = _rand_tiled(m, k, ta, DENSITY[da], rng)
    b = _rand_tiled(k, n, tb, DENSITY[db], rng)
    oA, oB = host.coo_to_csr(*a), host.coo_to_csr(*b)
    oC = host.spgemm(oA, oB)
    OA, OB = tiles.tile_format(*a), tiles.tile_format(*b)
    P = {keep: tiles.tiled_product(OA, OB, keep_empty=bool(keep)) for keep in (0, 1)}
    tA, tB = engine.convert_coo(*a), engine.convert_coo(*b)
    assert _dense(tA) == (da == "dense") and _dense(tB) == (db == "dense")
    assert engine.count_flop(tA, tB) == host.flop(oA, oB)
    seen = set()
    try:
        for path in PATHS:
            for step2 in range(4):
                for owner in range(5):
                    keep = (path + step2 + owner) % 2
                    tag = f"{shape} {da}x{db} path {path} step2 {step2} owner {owner} keep {keep}"
                    with Opts(engine, step1_path=path, step2_kernel=step2, owner=owner, keep_empty_tiles=keep):
                        if (step2 + owner) % 3 == 0:          # three panels
                            got, infos = _product(engine, tA, tB, 3)
                            assert all((i.rows, i.cols) == (m, n) for i in infos), tag
                            _assert_same(got, oC, tag)
                            continue
                        C = engine.step1(tA, tB)
                        Pk = P[keep]
                        i = C.info
                        assert (i.rows, i.cols, i.tiles, i.pairs) == (m, n, Pk.c_tile_col.size, Pk.pairs_a.size), tag
                        for name, want in (("row_ptr", Pk.c_row_ptr), ("tile_row", Pk.c_tile_row),
                                           ("tile_col", Pk.c_tile_col), ("pair_ptr", Pk.pair_ptr),
                                           ("pairs_a", Pk.pairs_a), ("pairs_b", Pk.pairs_b)):
                            assert np.array_equal(C.array(name), want), (tag, name)
                        engine.step2(tA, tB, C)
                        assert np.array_equal(C.array("masks").reshape(-1, 16), Pk.c_masks), tag
                        assert np.array_equal(C.array("tile_nnz_ptr"), Pk.c_tile_nnz_ptr), tag
                        engine.step3(tA, tB, C)
                        s3 = engine.last_step3_kernel
                        assert s3 == _expected_s3(owner, step2, da == "dense", db == "dense", C.info.nnz, C.info.pairs), tag
                        seen.add((path, step2, owner, s3))
                        _assert_same(C.to_coo(), oC, tag)
                        rp, cc, vv = C.to_csr()
                        assert np.array_equal(rp, oC.ptr) and np.array_equal(cc, oC.idx), tag
                        _assert_bits(vv, oC.val, tag)
                        C.free()
        # the automatic choices of this density combination ran end to end (spgemm, not the step calls)
        C = engine.spgemm(tA, tB)
        i = C.info
        assert (i.rows, i.cols) == (m, n) and C.array("tile_col").max() < -(-n // 16)
        assert engine.last_step3_kernel == _expected_s3(0, 0, da == "dense", db == "dense", i.nnz, i.pairs)
        _assert_same(C.to_coo(), oC)
        C.free()
    finally:
        tA.free(); tB.free()
    assert len({s for (_, _, _, s) in seen}) == 4


@gpu
@pytest.mark.parametrize("da,db", [("dense", "hyper"), ("hyper", "dense")])
def test_handle_roles_with_size_plans_and_graphs(engine, da, db):
    """A (m x k) and B (k x m) with the same handles in both roles, A*B then B*A, four rounds: views and row slices are
    cached per handle and role, size plans and graphs per operand pair.  Round 0 records, round 1 captures, later
    rounds replay; no size read-back stalls after round 0; every result bit-identical to the oracle."""
    m, k = 533, 1203
    rng = np.random.default_rng(77)
    a = _rand_tiled(m, k, 900, DENSITY[da], rng)
    b = _rand_tiled(k, m, 900, DENSITY[db], rng)
    oA, oB = host.coo_to_csr(*a), host.coo_to_csr(*b)
    want = {"AB": host.spgemm(oA, oB), "BA": host.spgemm(oB, oA)}
    tA, tB = engine.convert_coo(*a), engine.convert_coo(*b)
    engine.set_option(pem.OPT_SIZE_PLANS, 1)              # clears remembered sizes
    engine.set_option(pem.OPT_GRAPHS, 1)                  # drops the graphs
    try:
        for rnd in range(4):
            for name, X, Y, shape in (("AB", tA, tB, (m, m)), ("BA", tB, tA, (k, k))):
                s1, g1 = engine.size_stalls, engine.graph_replays
                C = engine.spgemm(X, Y)
                if rnd:
                    assert engine.size_stalls == s1, (rnd, name)
                assert engine.graph_replays - g1 == (0 if rnd == 0 else 1), (rnd, name)
                assert (C.info.rows, C.info.cols) == shape
                _assert_same(C.to_coo(), want[name], f"round {rnd} {name}")
                C.free()
        assert engine.count_flop(tA, tB) == host.flop(oA, oB) and engine.count_flop(tB, tA) == host.flop(oB, oA)
    finally:
        engine.set_option(pem.OPT_GRAPHS, 1)
        engine.set_option(pem.OPT_SIZE_PLANS, 1)
        tA.free(); tB.free()


def _sliced_products(A, B, keep):
    """Tile products counted by the row-sliced expansion: per A tile and occupied column c, the B tiles of B' row k
    whose row c is occupied."""
    TA, TB = tiles.tile_format(*A.coo()), tiles.tile_format(*B.coo())
    a_occ = np.bitwise_or.reduce(TA.masks, axis=1) if TA.cnt else np.zeros(0, np.uint16)
    b_occ = np.bitwise_or.reduce(TB.masks_t, axis=1) if TB.cnt else np.zeros(0, np.uint16)
    total = 0
    for t in range(TA.cnt):
        kk = TA.tile_col[t]
        occ = b_occ[TB.tile_row_ptr[kk]:TB.tile_row_ptr[kk + 1]].astype(np.int64)
        for c in range(16):
            if a_occ[t] >> c & 1:
                total += int(np.count_nonzero(occ >> c & 1))
    return total


def _run_constructed(engine, A, B, paths, owners=range(5), keeps=(0, 1), step2s=(0,), f32=False, check=None):
    """Every (path, owner, keep, step-2 kernel) combination on A*B against the oracle, bit for bit; check(info, path,
    owner, keep, step2) asserts the path indicators of each run."""
    _, _, oC = _oracle(A, B, f32)
    tA, tB = _convert(engine, A, f32), _convert(engine, B, f32)
    try:
        for path in paths:
            for owner in owners:
                if f32 and owner in (1, 3):
                    continue
                for keep in keeps:
                    for step2 in step2s:
                        tag = f"path {path} owner {owner} keep {keep} step2 {step2}"
                        with Opts(engine, step1_path=path, owner=owner, keep_empty_tiles=keep, step2_kernel=step2):
                            C = engine.spgemm(tA, tB)
                        try:
                            assert (C.info.rows, C.info.cols) == (A.rows, B.cols), tag
                            if check:
                                check(C.info, path, owner, keep, step2, tag)
                            _assert_same(C.to_coo(), oC, tag)
                        finally:
                            C.free()
    finally:
        tA.free(); tB.free()
    return oC


PAIR_COUNTS = [12, 13, 32, 33, 144, 145, 256, 257, 512, 513, 1024, 1025]


@gpu
@pytest.mark.parametrize("dense", [False, True])
@pytest.mark.parametrize("shift", [0, 31, 127])
@pytest.mark.parametrize("p", PAIR_COUNTS)
def test_pair_list_lengths_with_witnesses(engine, p, shift, dense):
    """C' tiles of p pairs at the pair-list thresholds, n and n+1: SORT_MAX 12 and WSORT_MAX 256 (per-row path),
    RS_GROUP_MAX 32 and the 64/128-thread row sort at 256 (row sort), RS_SMALL 1024 (row sort or radix sort, seen in
    last_sort_passes; with p = 1024 / 1025 also EX_CHUNK: 2048 / 2050 work items), S3C_NP 32 and SCAP 144 staged
    pairs.  Only RS_SMALL has an indicator; the others are compared on values.  (The per-row path's row thresholds,
    LARGE_LA, LARGE_P, HASH_MAXP and HASH_SPREAD, have cases of their own below: here p A tiles reach p products, so
    a row is heavy from p = 513 on and never hashes 1024 products.)  A shift tile of 31 or 127 pairs in front moves the list across 32-pair
    hit blocks and 128-pair step-2 blocks and step-3 windows.  The order witnesses sit in the first and last pairs;
    dense operands make step 2 run in dense-tile mode (no hit words) and step 3 the window kernel."""
    A, B = pair_family(p, shift, dense=dense)
    row = p + shift
    ad, bd = _is_dense(A), _is_dense(B)            # B's witness tiles hold 9 nonzeros: dense by the step-2 rule
    assert ad == dense and (bd or not dense)

    def check(info, path, owner, keep, step2, tag):
        assert info.pairs == row, tag
        passes = engine.last_sort_passes
        if path in (1, 5) or (path == 0):                  # small operands: the per-row path
            assert passes == -1, tag
        else:
            assert passes == (0 if row <= 1024 else 1), tag     # window 2 tile columns, 1 tile row: 1 + 1 key bits
            sliced = path == 4 and not keep
            assert info.tile_products == (_sliced_products(A, B, keep) if sliced else row), tag
        assert engine.last_step3_kernel == _expected_s3(owner, step2, ad, bd, info.nnz, info.pairs), tag

    oC = _run_constructed(engine, A, B, PATHS, step2s=(0, 3) if dense else (0,), check=check)
    v = oC.val
    assert np.isnan(v).sum() == 4 and np.isinf(v).sum() == 4 and np.any((v == 0) & np.signbit(v))


@gpu
@pytest.mark.parametrize("p", [33, 145, 1025])
def test_pair_list_witnesses_fp32(engine, p):
    """The fp32 instantiation on the same witnesses (2^-24, 2^127, 2^-149): subnormals survive (no FTZ), the sign of
    zero and the order of summation match the fp32 oracle bit for bit."""
    A, B = pair_family(p, 31, fmt=F32)
    for M in (A, B):
        for key, x in M.e.items():
            assert np.isnan(x) or float(np.float32(x)) == x, (key, x)            # exactly representable
    oC = _run_constructed(engine, A, B, PATHS, owners=(0, 2, 4), f32=True)
    assert np.any((oC.val != 0) & (np.abs(oC.val) < np.finfo(np.float32).smallest_normal))


@gpu
@pytest.mark.parametrize("width", [1 << 16, (1 << 16) + 1])
def test_small_operand_rule_reads_b_width(engine, width):
    """One A tile times B of 65536 / 65537 tile columns: the automatic step 1 takes the per-row path only while B
    has at most 65536 tile columns (a tiny A does not make the product small)."""
    A, B = window_case(width)

    def check(info, path, owner, keep, step2, tag):
        assert info.cols == B.cols and -(-B.cols // 16) == width, tag
        if path == 0:
            assert (engine.last_sort_passes == -1) == (width <= 65536), tag

    _run_constructed(engine, A, B, PATHS, owners=(0, 1, 2), keeps=(0,), check=check)


@gpu
@pytest.mark.parametrize("nb", [32768, 32769])
def test_small_operand_rule_counts_tiles(engine, nb):
    """A.tiles + B.tiles = 65536 / 65537 (B 32768 tile columns): per-row path only up to 65536 tiles."""
    A, B = diag_tiles_case(32768, nb)

    def check(info, path, owner, keep, step2, tag):
        if path == 0:
            assert (engine.last_sort_passes == -1) == (32768 + nb <= 65536), tag

    _run_constructed(engine, A, B, (0, 3), owners=(0,), keeps=(0,), check=check)


@gpu
@pytest.mark.parametrize("width,tile_rows,passes", [(8192, 1, 0), (8193, 1, 0),
                                                    (1 << 22, 1, 0), ((1 << 22) + 1, 1, 3),
                                                    ((1 << 22) + 1, 512, 4), ((1 << 22) + 1, 513, 5)])
def test_window_width_and_key_bits(engine, width, tile_rows, passes):
    """C' rows whose window is 8192 / 8193 tile columns (RS_BMW * 32: the row sort's counting path or its sorting
    network), 2^22 / 2^22 + 1 (the row sort needs wbits + 10 <= 32), and wbits = 23 with 512 / 513 tile rows
    (32 / 33 key bits: 32-bit or 64-bit keys, 4 or 5 radix passes)."""
    A, B = window_case(width, tile_rows)

    def check(info, path, owner, keep, step2, tag):
        assert engine.last_sort_passes == passes, tag
        assert info.cols == B.cols and info.tiles == 2 * tile_rows, tag

    _run_constructed(engine, A, B, (3, 4) + ((0,) if width > 65536 else ()), owners=(0, 1, 2, 3, 4), keeps=(0, 1), check=check)


@gpu
@pytest.mark.parametrize("kind,n", [("a_tiles", 512), ("products", 16384)])
def test_heavy_row_thresholds(engine, kind, n):
    """LARGE_LA (a row of more than 512 A tiles) and LARGE_P (more than 16384 tile products): the per-row path gives
    such a row 1024-thread count and fill kernels.  Beside a light companion row, which keeps the 128-thread kernels
    busy on both sides, the heavy side launches exactly two kernels more in step 1 than the side at n."""
    build = many_a_tiles_case if kind == "a_tiles" else heavy_row_case
    cases = {x: build(x) for x in (n, n + 1)}
    for path in (0, 1, 5):
        launches = {}
        for x, (A, B) in cases.items():
            tA, tB = _convert(engine, A), _convert(engine, B)
            try:
                with Opts(engine, step1_path=path):
                    l0 = engine.launch_count
                    C = engine.step1(tA, tB)
                    launches[x] = engine.launch_count - l0
                    assert engine.last_sort_passes == -1, (path, x)
                C.free()
            finally:
                tA.free(); tB.free()
        assert launches[n + 1] - launches[n] == 2, (path, launches)
    for x, (A, B) in cases.items():
        _, P, _ = _row_stats(A, B)[0]

        def check(info, path, owner, keep, step2, tag):
            if path == 3:
                assert info.tile_products == P + _row_stats(A, B)[1][1], tag

        _run_constructed(engine, A, B, PATHS, owners=(0, 2), keeps=(0,), check=check)


@gpu
@pytest.mark.parametrize("width", [20000, 1 << 20])
@pytest.mark.parametrize("P", [1024, 1025])
def test_hash_row_capacity(engine, P, width):
    """HASH_MAXP: a row of 4 A tiles and 1024 tile products fills the hash table's 2048 slots; 1025 products go to the
    bitmap.  Over a window of 2^20 tile columns the bitmap does not fit shared memory, so both per-row paths (5: hash
    on request, 1: because the window is wide) multiply the 1024-product row and refuse the 1025-product one with
    PEM_ERR_LIMIT, which shows the side that ran; expand-sort-compress multiplies both.  Over 20000 tile columns every
    path multiplies both sides."""
    A, B = hash_row_case(P, width)
    wide = width > 65536
    if wide:
        tA, tB = _convert(engine, A), _convert(engine, B)
        try:
            for path in (1, 5):
                with Opts(engine, step1_path=path):
                    if P <= 1024:
                        engine.spgemm(tA, tB).free()
                    else:
                        with pytest.raises(pem.PemError) as e:
                            engine.spgemm(tA, tB)
                        assert e.value.code == -5, path
        finally:
            tA.free(); tB.free()

    def check(info, path, owner, keep, step2, tag):
        assert info.pairs == P, tag
        per_row = path in (1, 5) or (path == 0 and not wide)
        assert (engine.last_sort_passes == -1) == per_row, tag

    paths = ((0, 3, 4) + ((1, 5) if P <= 1024 else ())) if wide else PATHS
    _run_constructed(engine, A, B, paths, owners=(0, 2), keeps=(0, 1), check=check)


@gpu
@pytest.mark.parametrize("jmax", [1023, 1024])
def test_hash_spread_rule(engine, jmax):
    """HASH_SPREAD: 64 tile products over 32 / 33 bitmap words; under the automatic choice (paths 0 and 1) the row
    takes the hash table only when the window holds more than 16 tile columns per product.  Nothing the engine
    reports tells the two accumulators apart here, so this case is compared on values; its CPU self-check keeps it
    straddling the rule."""
    A, B = spread_case(jmax)

    def check(info, path, owner, keep, step2, tag):
        assert info.pairs == 64 and (engine.last_sort_passes == -1) == (path in (0, 1, 5)), tag

    _run_constructed(engine, A, B, (0, 1, 5, 3), owners=(0, 2), keeps=(0, 1), check=check)


@gpu
@pytest.mark.parametrize("a_short,b_short,kernel", [(0, 0, 4), (1, 0, 2), (0, 1, 2)])
def test_step2_dense_rule_at_eight_per_tile(engine, a_short, b_short, kernel):
    """A.nnz = 8 * A.tiles (row-mask form) against one less (list form), and the same for B: only when both are
    dense does step 2 drop the hit words, which the automatic step 3 shows by taking the window kernel."""
    A, B = step2_form_case(a_short, b_short)

    def check(info, path, owner, keep, step2, tag):
        assert (info.pairs, info.nnz) == (3, 8), tag
        if owner == 0 and step2 == 0:
            assert engine.last_step3_kernel == kernel, tag

    _run_constructed(engine, A, B, PATHS, owners=(0, 2, 4), keeps=(0, 1), step2s=(0, 1, 2, 3), check=check)


@gpu
@pytest.mark.parametrize("nnz,kernel", [(3, 2), (4, 4)])
def test_step3_window_rule_at_four_entries_per_pair(engine, nnz, kernel):
    """nnz(C) = 4 * pairs takes the window kernel, one entry less the entry-owner kernel (with hit words)."""
    A, B = entries_per_pair_case(nnz)

    def check(info, path, owner, keep, step2, tag):
        assert (info.pairs, info.nnz) == (1, nnz), tag
        if owner == 0:
            assert engine.last_step3_kernel == kernel, tag

    _run_constructed(engine, A, B, PATHS, owners=(0, 1, 2, 3, 4), keeps=(0,), check=check)


@gpu
@pytest.mark.parametrize("n_empty", [510, 511])
def test_entry_owner_block_spanning_empty_tiles(engine, n_empty):
    """keep-empty: the entry-owner kernel's first 128-entry block spans n_empty + 2 = 512 / 513 C' tiles (S3E_TMAX:
    tile offsets staged in shared memory up to 512)."""
    A, B = empty_span_case(n_empty)

    def check(info, path, owner, keep, step2, tag):
        assert info.tiles == (n_empty + 2 if keep else 2), tag
        assert info.nnz == 224, tag

    _run_constructed(engine, A, B, (0, 1, 3), owners=(0, 2, 3, 4), keeps=(0, 1), check=check)


@gpu
@pytest.mark.parametrize("seed", [1, 2])
def test_special_values_in_random_operands(engine, seed):
    """Random independent operands with +-0.0, subnormals, +-Inf and NaN written into chosen positions of A and B,
    and Infs of B opposite explicit zeros of A: every step-1 path and step-3 owner, values bit for bit, NaN and
    Inf exactly where the oracle has them."""
    rng = np.random.default_rng(seed)
    a = list(_rand_tiled(61, 700, 120, (1, 12), rng))
    b = list(_rand_tiled(700, 3011, 900, (1, 12), rng))
    specials = np.array([0.0, -0.0, 5e-324, -5e-324, 2.2250738585072009e-308, 2.0 ** 1023, -(2.0 ** 1023),
                         2.0 ** -600, -(2.0 ** -600), np.inf, -np.inf, np.nan])
    for M in (a, b):
        V = M[4]
        at = rng.choice(V.size, size=V.size // 6, replace=False)
        V[at] = specials[rng.integers(0, specials.size - 3, at.size)]          # no Inf/NaN yet
        at = rng.choice(V.size, size=4, replace=False)
        V[at] = specials[[9, 10, 11, 9]]
    # an Inf in B row k opposite an explicit 0.0 in A column k
    ks = np.intersect1d(a[3], b[2])[:5]
    for kk in ks:
        a[4][np.flatnonzero(a[3] == kk)[0]] = 0.0
        b[4][np.flatnonzero(b[2] == kk)[0]] = np.inf
    A, B = Mat(61, 700), Mat(700, 3011)
    for M, (_, _, I, J, V) in ((A, a), (B, b)):
        for i, j, x in zip(I, J, V):
            M.put(i, j, float(x))
    oC = _run_constructed(engine, A, B, PATHS, owners=range(5), keeps=(0, 1))
    assert np.isnan(oC.val).any() and np.isinf(oC.val).any()
