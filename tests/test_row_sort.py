"""Step 1's row sort (expand-sort-compress with every C' row of at most 1024 pairs): one warp orders one C' row, and
the rows of one block are independent.  The constructed products put rows of very different lengths next to each
other: empty rows, rows of one pair, rows at and around the 32-pair steps of the warp, C' tiles of far more than 32 pairs
(one group of the counting scatter) and rows whose window is wider than the 8192-column bitmap (the sorting network),
so the rows that share a block take different paths and leave at different times.  C' structure and pair lists are
compared with the tile oracle, values bit for bit with the host oracle."""
import numpy as np
import pytest

import pem_spgemm_b200 as pem
from oracle import host, tiles

gpu = pytest.mark.gpu

BITMAP_COLUMNS = 8192


def mixed_rows(lengths, seed):
    """A (16 * R rows) times B: C' row i holds exactly lengths[i] pairs.  Every row has tile rows of B of its own
    (tile index K), so rows do not share pairs.  A tile (i, K) has a nonzero in local column 0 and every B tile
    (K, J) one in local row 0, so every reachable pair is kept.  A row draws the tile columns J of its B rows from a
    pool: a small pool makes large C' tiles, a large one many small tiles; a row whose length is given as negative
    spreads its pool over more than the bitmap's window."""
    rng = np.random.default_rng(seed)
    rows_of = []                                   # per C' row: the J lists of its B tile rows
    for i, n in enumerate(lengths):
        wide = n < 0
        n = abs(n)
        if wide:
            pool = np.unique(np.concatenate([[0, BITMAP_COLUMNS + 100], rng.integers(0, BITMAP_COLUMNS + 100, 20)]))
        else:
            pool = np.arange((3, 12, 60, 400)[i % 4])
        Ks, left = [], n
        if wide:                                   # the row's window for sure: its first and last pool column
            Ks.append(pool[[0, -1]])
            left -= 2
        while left:
            s = min(left, int(rng.integers(1, min(len(pool), 40) + 1)))
            Ks.append(np.sort(rng.choice(pool, size=s, replace=False)))
            left -= s
        rows_of.append(Ks)
    nk = sum(len(Ks) for Ks in rows_of)
    ncols = 16 * (max([int(j.max()) for Ks in rows_of for j in Ks], default=0) + 1)
    AI, AJ, BI, BJ = [], [], [], []
    K = 0
    for i, Ks in enumerate(rows_of):
        for js in Ks:
            AI.append(16 * i + rng.integers(0, 16, 2)); AJ.append(np.array([16 * K, 16 * K]))
            BI.append(np.full(js.size, 16 * K)); BJ.append(16 * js + rng.integers(0, 16, js.size))
            K += 1
    cat = lambda x: np.concatenate(x).astype(np.int32) if x else np.zeros(0, np.int32)
    AI, AJ, BI, BJ = cat(AI), cat(AJ), cat(BI), cat(BJ)
    A = _coo(16 * len(lengths), 16 * max(nk, 1), AI, AJ, rng)
    B = _coo(16 * max(nk, 1), ncols, BI, BJ, rng)
    return A, B


def _coo(rows, cols, I, J, rng):
    key = np.unique(I.astype(np.int64) * cols + J)
    I, J = (key // cols).astype(np.int32), (key % cols).astype(np.int32)
    return rows, cols, I, J, rng.uniform(-1, 1, I.size)


SHORT = [0, 1, 31, 32, 33, 0, 227, 64, 5, 0, 0, 255, 256, 120, -40, 17, 96, 0, 2, 250, -256, 33, 1, 0]
LONG = [1024, 0, 1, 1000, -1024, 513, 0, 700, 31, 257, -300, 0, 1024, 2, 999]


@pytest.mark.parametrize("lengths", [SHORT, LONG])
def test_mixed_rows_have_the_claimed_lengths(lengths):
    A, B = mixed_rows(lengths, seed=len(lengths))
    P = tiles.tiled_product(tiles.tile_format(*A), tiles.tile_format(*B), keep_empty=False)
    per_row = np.bincount(P.c_tile_row, weights=np.diff(P.pair_ptr), minlength=len(lengths)).astype(int)
    assert list(per_row) == [abs(n) for n in lengths]
    for i, n in enumerate(lengths):
        cols = P.c_tile_col[P.c_tile_row == i]
        if n:
            assert (cols.max() - cols.min() + 1 > BITMAP_COLUMNS) == (n < 0), i
    sizes = np.diff(P.pair_ptr)
    assert sizes.max() > 32                    # a C' tile (one group of the scatter) of more than 32 pairs


@gpu
@pytest.mark.parametrize("variant", [0, 1])
@pytest.mark.parametrize("path", [3, 4])
@pytest.mark.parametrize("lengths", [SHORT, LONG], ids=["short", "long"])
def test_row_sort_mixed_rows(engine, lengths, path, variant):
    """Rows of mixed lengths and paths in one block, through the tile-level and the row-sliced expansion, written
    in one pass or counted first (PEM_OPT_ESC_VARIANT bit 0)."""
    A, B = mixed_rows(lengths, seed=len(lengths))
    P = tiles.tiled_product(tiles.tile_format(*A), tiles.tile_format(*B), keep_empty=False)
    oC = host.spgemm(host.coo_to_csr(*A), host.coo_to_csr(*B))
    tA, tB = engine.convert_coo(*A), engine.convert_coo(*B)
    engine.set_option(pem.OPT_STEP1_PATH, path)
    engine.set_option(pem.OPT_ESC_VARIANT, variant)
    try:
        C = engine.step1(tA, tB)
        assert engine.last_sort_passes == 0
        i = C.info
        assert (i.tiles, i.pairs) == (P.c_tile_col.size, P.pairs_a.size)
        for name, want in (("row_ptr", P.c_row_ptr), ("tile_row", P.c_tile_row), ("tile_col", P.c_tile_col),
                           ("pair_ptr", P.pair_ptr), ("pairs_a", P.pairs_a), ("pairs_b", P.pairs_b)):
            assert np.array_equal(C.array(name), want), name
        engine.step2(tA, tB, C)
        engine.step3(tA, tB, C)
        r, c, v = C.to_coo()
        ro, co, vo = oC.to_coo()
        assert np.array_equal(r, ro) and np.array_equal(c, co)
        assert np.array_equal(v.view(np.uint64), vo.view(np.uint64))
        C.free()
    finally:
        engine.set_option(pem.OPT_STEP1_PATH, 0)
        engine.set_option(pem.OPT_ESC_VARIANT, 0)
        tA.free(); tB.free()
