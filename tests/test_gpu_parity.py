"""GPU parity tests (run with -m gpu on a B200): the CUDA engine, called through the C ABI,
against the host oracle on identical seeded inputs.  Structure and indices must be bit-exact;
values are compared bit-exact as well (the engine keeps the oracle's ascending-k fma order),
with the north-star tolerance 1e-12 as the stated bound for floating point."""
import numpy as np
import pytest

import pem_spgemm_b200 as pem
from oracle import host, tiles
from pem_spgemm_b200 import synth

pytestmark = pytest.mark.gpu
RTOL = 1e-12  # north_star tolerance for fp64 values


def _assert_bits(v, vo, tag=""):
    """Bit equality of two value arrays: the sign of zero counts, and a NaN matches any NaN (payloads
    legitimately differ between the host and the GPU).  np.array_equal would take -0.0 for +0.0 and fail on NaN."""
    v, vo = np.asarray(v), np.asarray(vo)
    assert v.dtype == vo.dtype and v.shape == vo.shape, (v.dtype, vo.dtype, v.shape, vo.shape)
    u = np.uint32 if v.dtype == np.float32 else np.uint64
    if np.array_equal(v.view(u), vo.view(u)):
        return
    nan, nano = np.isnan(v), np.isnan(vo)
    assert np.array_equal(nan, nano), f"{tag} NaN at {np.flatnonzero(nan != nano)[:10]}"
    bad = np.flatnonzero((v.view(u) != vo.view(u)) & ~nan)
    assert bad.size == 0, f"{tag} {bad.size} values differ in their bits, first at {bad[:10]}: {v[bad[:5]]} vs {vo[bad[:5]]}"


def _assert_same_C(Cres, Coracle, exact=True):
    r, c, v = Cres.to_coo()
    ro, co, vo = Coracle.to_coo()
    assert r.size == ro.size
    assert np.array_equal(r, ro) and np.array_equal(c, co)          # structure: bit-exact
    np.testing.assert_allclose(v, vo, rtol=RTOL, atol=0)            # the stated tolerance
    if exact:
        _assert_bits(v, vo)                                          # same fma order => same bits


def _check_tiled(T, O):
    i = T.info
    assert (i.rows, i.cols, i.tile_rows, i.tile_cols, i.tiles) == (O.rows, O.cols, O.tile_rows, O.tile_cols, O.cnt)
    assert np.array_equal(T.array("tile_nnz_ptr").astype(np.int64), O.tile_nnz_ptr)
    assert np.array_equal(T.array("vals"), O.vals)
    assert np.array_equal(T.array("masks").reshape(-1, 16), O.masks)
    assert np.array_equal(T.array("masks_t").reshape(-1, 16), O.masks_t)
    assert np.array_equal(T.array("row_ptr").reshape(-1, 16), O.row_ptr)
    assert np.array_equal(T.array("row_col_idx"), O.row_col_idx)
    assert np.array_equal(T.array("tile_row_ptr"), O.tile_row_ptr)
    assert np.array_equal(T.array("tile_col_idx"), O.tile_col)
    assert np.array_equal(T.array("tile_row_idx"), O.tile_row)
    z = np.zeros(0, np.uint16)
    assert np.array_equal(T.array("col_occ"), np.bitwise_or.reduce(O.masks, axis=1) if O.cnt else z)
    assert np.array_equal(T.array("row_occ"), np.bitwise_or.reduce(O.masks_t, axis=1) if O.cnt else z)


SHAPES = [((50, 70), 400, 11), ((16, 16), 256, 4), ((1, 1), 1, 1), ((333, 333), 5000, 2),
          ((17, 4000), 3000, 3), ((4000, 17), 3000, 5), ((1000, 1000), 1, 6)]


@pytest.mark.parametrize("shape,nnz,seed", SHAPES)
@pytest.mark.parametrize("transpose", [False, True])
def test_conversion_matches_tile_oracle(engine, shape, nnz, seed, transpose):
    rows, cols, I, J, V = synth.random_sparse(*shape, nnz, seed=seed)
    T = engine.convert_coo(rows, cols, I, J, V, transpose=transpose)
    _check_tiled(T, tiles.tile_format(rows, cols, I, J, V, transpose=transpose))
    T.free()


def test_dense_blocks_all_step3_variants(engine):
    """Fully dense 16x16 tiles (256 nonzeros per C tile: eight passes of a warp in the tile-class kernel,
    two whole blocks of the entry-owner one) and a ragged dense matrix."""
    for n in (32, 40):
        I, J = np.divmod(np.arange(n * n, dtype=np.int32), n)
        V = np.random.default_rng(n).uniform(-1, 1, n * n)
        _, _, oC = host.spgemm_from_coo(n, n, I, J, V, False)
        A = engine.convert_coo(n, n, I, J, V)
        for owner in (0, 1, 2, 3, 4):
            engine.set_option(pem.OPT_OWNER, owner)
            try:
                C = engine.spgemm(A, A)
                _assert_same_C(C, oC)
                C.free()
            finally:
                engine.set_option(pem.OPT_OWNER, 0)
        A.free()


@pytest.mark.parametrize("owner,step2", [(0, 0), (4, 0), (4, 3), (2, 0), (0, 1)])
def test_dense_tiles_with_long_pair_lists(engine, owner, step2):
    """A wide matrix with dense tiles times its transpose: every C' tile owns 375 pairs, more than the window kernel
    stages (144), so its nonzeros take the kernel's unstaged path: a walk over all pairs in dense-tile mode (step 2
    automatic: no hit words are produced), the hit blocks when the row-mask form is forced or the entry-owner kernel asked for."""
    rows, cols, I, J, V = synth.random_sparse(48, 6000, 40000, seed=21)
    _, _, oC = host.spgemm_from_coo(rows, cols, I, J, V, True)
    A = engine.convert_coo(rows, cols, I, J, V)
    B = engine.transpose(A)
    assert A.info.nnz >= 8 * A.info.tiles
    engine.set_option(pem.OPT_OWNER, owner)
    engine.set_option(pem.OPT_STEP2_KERNEL, step2)
    try:
        for _ in range(3):                            # ordinary, captured, graph launch
            C = engine.spgemm(A, B)
            assert C.info.pairs == 9 * 375
            assert engine.last_step3_kernel == (2 if owner == 2 or (owner == 0 and step2 == 1 and C.info.nnz < 4 * C.info.pairs) else 4)
            _assert_same_C(C, oC)
            C.free()
    finally:
        engine.set_option(pem.OPT_OWNER, 0)
        engine.set_option(pem.OPT_STEP2_KERNEL, 0)
    B.free(); A.free()


@pytest.mark.parametrize("shape,nnz,seed", SHAPES + [((16, 16), 0, 9)])
def test_device_transpose_equals_transposed_conversion(engine, shape, nnz, seed):
    """pem_tiled_transpose (A^T from A's tiles) must reproduce pem_convert_coo(transpose=1) array by array."""
    rows, cols, I, J, V = synth.random_sparse(*shape, nnz, seed=seed)
    A = engine.convert_coo(rows, cols, I, J, V)
    T = engine.transpose(A)
    _check_tiled(T, tiles.tile_format(rows, cols, I, J, V, transpose=True))
    if I.size:
        C = engine.spgemm(A, T)
        _, _, oC = host.spgemm_from_coo(rows, cols, I, J, V, True)
        _assert_same_C(C, oC)
        C.free()
    T.free(); A.free()


@pytest.mark.parametrize("shape,nnz,seed", SHAPES + [((40, 40), 0, 3)])
@pytest.mark.parametrize("where", ["host", "device"])
def test_csr_in_and_csr_out(engine, shape, nnz, seed, where):
    """pem_convert_csr must build the same tiled arrays as the COO path, and pem_result_to_csr must return the
    oracle's CSR of C = A*A^T (row pointer, ascending columns, value bits)."""
    import torch
    rows, cols, I, J, V = synth.random_sparse(*shape, nnz, seed=seed)
    oA = host.coo_to_csr(rows, cols, I, J, V)
    rp = oA.ptr.astype(np.int32)
    rng = np.random.default_rng(seed)
    cj, cv = oA.idx.copy(), oA.val.copy()
    for r in range(rows):                                   # columns need not be sorted inside a row
        b, e = rp[r], rp[r + 1]
        p = rng.permutation(e - b)
        cj[b:e], cv[b:e] = cj[b:e][p], cv[b:e][p]
    if where == "device":
        keep = [torch.from_numpy(x).cuda() for x in (rp, cj, cv)]
        torch.cuda.synchronize()
        A = engine.convert_csr(rows, cols, *(t.data_ptr() for t in keep))
    else:
        A = engine.convert_csr(rows, cols, rp, cj, cv)
    _check_tiled(A, tiles.tile_format(rows, cols, I, J, V))
    T = engine.convert_csr(rows, cols, rp, cj, cv, transpose=True)
    _check_tiled(T, tiles.tile_format(rows, cols, I, J, V, transpose=True))
    C = engine.spgemm(A, T)
    _, _, oC = host.spgemm_from_coo(rows, cols, I, J, V, True)
    crp, cc, cvv = C.to_csr()
    assert np.array_equal(crp, oC.ptr) and np.array_equal(cc, oC.idx) and np.array_equal(cvv, oC.val)
    C.free(); T.free(); A.free()


@pytest.mark.parametrize("k", [1, 2, 3, 4, 5])
def test_fp32_instantiation_matches_fp32_oracle(engine, k):
    """SURVEY.md section 8f rank 4: the second value type.  fp32 operands, single-precision fma in the same
    ascending-k order: structure identical to the fp64 product, value bits equal to the fp32 oracle's."""
    name, tb, (rows, cols, I, J, V) = synth.config(k, small=True)
    V32 = V.astype(np.float32)
    A = engine.convert_coo(rows, cols, I, J, V32, dtype=np.float32)
    assert A.dtype == np.float32
    O = tiles.tile_format(rows, cols, I, J, V32.astype(np.float64))
    assert np.array_equal(A.array("vals"), O.vals.astype(np.float32))
    assert np.array_equal(A.array("masks").reshape(-1, 16), O.masks)
    B = engine.transpose(A) if tb else A
    oA = host.coo_to_csr(rows, cols, I, J, V32.astype(np.float64))
    oB = host.transpose(oA) if tb else oA
    oC = host.spgemm_f32(oA, oB)
    bounds = engine.partition_panels(A, B, 2)
    parts = []
    for p in range(2):
        C = engine.spgemm(A, B, panel=(bounds[p], bounds[p + 1]))
        assert C.dtype == np.float32
        parts.append(C.to_coo())
        if p == 0:
            s, a = C.checksum()
            np.testing.assert_allclose([s, a], [parts[0][2].astype(np.float64).sum(), np.abs(parts[0][2].astype(np.float64)).sum()],
                                       rtol=1e-9, atol=1e-9)
        C.free()
    r = np.concatenate([x[0] for x in parts]); c = np.concatenate([x[1] for x in parts]); v = np.concatenate([x[2] for x in parts])
    ro, co, vo = oC.to_coo()
    assert v.dtype == np.float32 and np.array_equal(r, ro) and np.array_equal(c, co)
    np.testing.assert_allclose(v, vo, rtol=1e-5, atol=0)             # stated fp32 tolerance
    _assert_bits(v, vo)                                              # same fma order => same bits
    # mixing value types and the fp64-only kernels are refused, not silently converted
    A64 = engine.convert_coo(rows, cols, I, J, V)
    with pytest.raises(pem.PemError):
        engine.spgemm(A64 if not tb else A, A if not tb else engine.transpose(A64))
    engine.set_option(pem.OPT_OWNER, 3)
    try:
        with pytest.raises(pem.PemError):
            engine.spgemm(A, B)
    finally:
        engine.set_option(pem.OPT_OWNER, 0)
    A64.free()
    if B is not A:
        B.free()
    A.free()


def test_conversion_dense_tile_and_empty(engine):
    I, J = np.divmod(np.arange(256, dtype=np.int32), 16)
    V = np.arange(256, dtype=np.float64)
    T = engine.convert_coo(16, 16, I, J, V)
    assert T.array("row_ptr")[-1] == 240 and np.all(T.array("masks") == 0xFFFF)
    T.free()
    z = np.zeros(0, np.int32)
    E = engine.convert_coo(40, 40, z, z, np.zeros(0))
    assert E.info.tiles == 0 and np.all(E.array("tile_row_ptr") == 0)
    C = engine.spgemm(E, E)
    assert C.info.nnz == 0 and C.info.tiles == 0
    assert C.to_coo()[0].size == 0
    C.free(); E.free()


def test_conversion_input_errors(engine):
    I = np.array([0, 0], np.int32); J = np.array([1, 1], np.int32)
    with pytest.raises(pem.PemError) as e:
        engine.convert_coo(4, 4, I, J, np.ones(2))
    assert e.value.code == -4
    with pytest.raises(pem.PemError) as e:
        engine.convert_coo(4, 4, np.array([4], np.int32), np.array([0], np.int32), np.ones(1))
    assert e.value.code == -3
    rows, cols, I, J, V = synth.random_sparse(10, 30, 50, seed=1)
    A = engine.convert_coo(rows, cols, I, J, V)
    with pytest.raises(pem.PemError) as e:       # rectangular A*A is rejected (spgemm.cu:782-786)
        engine.spgemm(A, A)
    assert e.value.code == -2
    A.free()


# 3: expand-sort-compress at tile level, 4: ... through B's row slices, 1: windowed bitmap SPA (0/2 pick one of them)
@pytest.mark.parametrize("step1_path", [3, 4, 1, 5])
@pytest.mark.parametrize("keep_empty", [1, 0])
@pytest.mark.parametrize("k", [1, 2, 3, 4, 5])
def test_steps_match_tile_oracle(engine, k, keep_empty, step1_path):
    """Step-by-step parity of C' structure, ordered pair lists, C masks and per-tile nnz."""
    name, tb, (rows, cols, I, J, V) = synth.config(k, small=True)
    engine.set_option(pem.OPT_KEEP_EMPTY_TILES, keep_empty)
    engine.set_option(pem.OPT_STEP1_PATH, step1_path)
    try:
        A = engine.convert_coo(rows, cols, I, J, V)
        B = engine.convert_coo(rows, cols, I, J, V, transpose=tb)
        OA = tiles.tile_format(rows, cols, I, J, V)
        OB = tiles.tile_format(rows, cols, I, J, V, transpose=tb)
        P = tiles.tiled_product(OA, OB, keep_empty=bool(keep_empty))
        C = engine.step1(A, B)
        info = C.info
        assert (info.tiles, info.pairs) == (P.c_tile_col.size, P.pairs_a.size)
        assert np.array_equal(C.array("row_ptr"), P.c_row_ptr)
        assert np.array_equal(C.array("tile_row"), P.c_tile_row)
        assert np.array_equal(C.array("tile_col"), P.c_tile_col)
        assert np.array_equal(C.array("pair_ptr"), P.pair_ptr)
        assert np.array_equal(C.array("pairs_a"), P.pairs_a)
        assert np.array_equal(C.array("pairs_b"), P.pairs_b)
        engine.step2(A, B, C)
        assert np.array_equal(C.array("masks").reshape(-1, 16), P.c_masks)
        assert np.array_equal(C.array("tile_nnz_ptr"), P.c_tile_nnz_ptr)
        # rowColIdx: (r<<4)|c of every set mask bit, tile by tile, row-major (spgemm.cu:582-587)
        t, r = np.nonzero(P.c_masks)
        bits = (P.c_masks[t, r].astype(np.int64)[:, None] >> np.arange(16)) & 1
        idx, cc = np.nonzero(bits)
        want = ((r[idx] << 4) | cc).astype(np.uint8)
        assert np.array_equal(C.array("row_col_idx"), want)
        engine.step3(A, B, C)
        _, _, Co = host.spgemm_from_coo(rows, cols, I, J, V, tb)
        _assert_same_C(C, Co)
        C.free(); A.free(); B.free()
    finally:
        engine.set_option(pem.OPT_KEEP_EMPTY_TILES, 0)
        engine.set_option(pem.OPT_STEP1_PATH, 0)


@pytest.mark.parametrize("shape,nnz,seed", SHAPES)
def test_spgemm_aat_random(engine, shape, nnz, seed):
    rows, cols, I, J, V = synth.random_sparse(*shape, nnz, seed=seed)
    A = engine.convert_coo(rows, cols, I, J, V)
    B = engine.convert_coo(rows, cols, I, J, V, transpose=True)
    C = engine.spgemm(A, B)
    oA, oB, oC = host.spgemm_from_coo(rows, cols, I, J, V, True)
    _assert_same_C(C, oC)
    assert engine.count_flop(A, B) == host.flop(oA, oB)
    s, a = C.checksum()
    np.testing.assert_allclose([s, a], [oC.val.sum(), np.abs(oC.val).sum()], rtol=1e-9, atol=1e-9)
    C.free(); A.free(); B.free()


def test_structural_zero_kept(engine):
    I = np.array([0, 0, 1, 1], np.int32); J = np.array([0, 1, 0, 1], np.int32)
    A = engine.convert_coo(2, 2, I, J, np.array([1.0, 1.0, 1.0, -1.0]))
    C = engine.spgemm(A, A)
    r, c, v = C.to_coo()
    assert list(v) == [2.0, 0.0, 0.0, 2.0]
    C.free(); A.free()


def test_config1_full_known_answers(engine):
    """Config 1 at full size against the pinned numbers of SURVEY.md section 8c."""
    rows, cols, I, J, V = synth.laplacian2d(256)
    A = engine.convert_coo(rows, cols, I, J, V)
    assert A.info.tiles == 19_936 and A.info.tile_rows == 4_096
    assert engine.count_flop(A, A) == 1_629_192
    engine.set_option(pem.OPT_KEEP_EMPTY_TILES, 1)
    C = engine.spgemm(A, A)
    engine.set_option(pem.OPT_KEEP_EMPTY_TILES, 0)
    assert (C.info.tiles, C.info.pairs, C.info.nnz) == (50_532, 97_512, 846_852)
    C.free()
    C = engine.spgemm(A, A)
    assert (C.info.tiles, C.info.nnz) == (43_364, 846_852)
    assert C.checksum() == (1032.0, 4_178_952.0)
    _, _, oC = host.spgemm_from_coo(rows, cols, I, J, V, False)
    _assert_same_C(C, oC)
    C.free(); A.free()


@pytest.mark.parametrize("k,nparts", [(2, 3), (4, 8), (3, 2)])
def test_panels_concatenate_to_full_result(engine, k, nparts):
    name, tb, (rows, cols, I, J, V) = synth.config(k, small=True)
    A = engine.convert_coo(rows, cols, I, J, V)
    B = engine.convert_coo(rows, cols, I, J, V, transpose=tb)
    bounds = engine.partition_panels(A, B, nparts)
    assert bounds[0] == 0 and bounds[-1] == A.info.tile_rows and np.all(np.diff(bounds) >= 0)
    _, _, oC = host.spgemm_from_coo(rows, cols, I, J, V, tb)
    parts = []
    for p in range(nparts):
        C = engine.spgemm(A, B, panel=(bounds[p], bounds[p + 1]))
        parts.append(C.to_coo()); C.free()
    r = np.concatenate([x[0] for x in parts]); c = np.concatenate([x[1] for x in parts])
    v = np.concatenate([x[2] for x in parts])
    ro, co, vo = oC.to_coo()
    assert np.array_equal(r, ro) and np.array_equal(c, co) and np.array_equal(v, vo)
    A.free(); B.free()


@pytest.mark.parametrize("k", [2, 3, 4])
def test_async_values_conversion(engine, k):
    """PEM_OPT_ASYNC_VALUES: pem_convert_coo returns while the values are still uploading from pinned host
    memory; the product (whose steps 1-2 overlap the upload), the accessors, the transpose and an early free
    must all see finished values."""
    import torch
    name, tb, (rows, cols, I, J, V) = synth.config(k, small=True)
    tI = torch.from_numpy(I.copy()).pin_memory(); tJ = torch.from_numpy(J.copy()).pin_memory(); tV = torch.from_numpy(V.copy()).pin_memory()
    _, _, oC = host.spgemm_from_coo(rows, cols, I, J, V, tb)
    engine.set_option(pem.OPT_ASYNC_VALUES, 1)
    try:
        for rep in range(3):
            A = engine.convert_coo(rows, cols, tI.numpy(), tJ.numpy(), tV.numpy())
            if rep == 0:
                B = engine.transpose(A) if tb else A
                C = engine.spgemm(A, B)
                _assert_same_C(C, oC)
                C.free()
                if B is not A:
                    B.free()
            elif rep == 1:
                assert np.array_equal(A.array("vals"), tiles.tile_format(rows, cols, I, J, V).vals)
                A.values_ready()
            A.free()                       # rep 2: freed with the upload possibly still in flight
    finally:
        engine.set_option(pem.OPT_ASYNC_VALUES, 0)


def test_device_pointer_input_and_pool_reuse(engine):
    import torch
    rows, cols, I, J, V = synth.random_sparse(2000, 2000, 30000, seed=8)
    dI = torch.from_numpy(I).cuda(); dJ = torch.from_numpy(J).cuda(); dV = torch.from_numpy(V).cuda()
    torch.cuda.synchronize()
    A = engine.convert_coo(rows, cols, dI.data_ptr(), dJ.data_ptr(), dV.data_ptr(), nnz=I.size)
    _check_tiled(A, tiles.tile_format(rows, cols, I, J, V))
    _, _, oC = host.spgemm_from_coo(rows, cols, I, J, V, False)
    for _ in range(3):                      # repeated products recycle pool memory
        C = engine.spgemm(A, A)
        _assert_same_C(C, oC)
        C.free()
    A.free()


@pytest.mark.parametrize("k", [1, 2, 3, 4, 5])
@pytest.mark.parametrize("step1_path", [0, 1, 2, 5])
def test_size_plans_replay_without_stalls(engine, k, step1_path):
    """PEM_OPT_SIZE_PLANS: the first product of an operand pair stalls at its size read-backs (the reference's
    spgemm.cu:1169, 1246, 1291) and records them; repeats of the same handles (whole product and panels) replay the
    sizes, stall nowhere before their final synchronisation and give the same bits; other operands get their own plan."""
    name, tb, (rows, cols, I, J, V) = synth.config(k, small=True)
    A = engine.convert_coo(rows, cols, I, J, V)
    B = engine.convert_coo(rows, cols, I, J, V, transpose=tb)
    _, _, oC = host.spgemm_from_coo(rows, cols, I, J, V, tb)
    engine.set_option(pem.OPT_STEP1_PATH, step1_path)
    engine.set_option(pem.OPT_SIZE_PLANS, 1)          # also clears the remembered sizes
    try:
        s0 = engine.size_stalls
        C = engine.spgemm(A, B)
        first = engine.size_stalls - s0
        assert first >= 3
        _assert_same_C(C, oC)
        C.free()
        for _ in range(3):
            s1 = engine.size_stalls
            C = engine.spgemm(A, B)
            assert engine.size_stalls == s1           # replayed
            _assert_same_C(C, oC)
            C.free()
        bounds = engine.partition_panels(A, B, 2)
        for rep in range(2):
            s1 = engine.size_stalls
            parts = [engine.spgemm(A, B, panel=(int(bounds[i]), int(bounds[i + 1]))) for i in range(2)]
            assert (engine.size_stalls == s1) == (rep == 1)
            assert sum(p.info.nnz for p in parts) == oC.nnz
            for p_ in parts:
                p_.free()
        # a second conversion of the same matrix is a different handle: its own plan, recorded again
        A2 = engine.convert_coo(rows, cols, I, J, V)
        s1 = engine.size_stalls
        C = engine.spgemm(A2, B)
        assert engine.size_stalls - s1 == first
        _assert_same_C(C, oC)
        C.free(); A2.free()
        engine.set_option(pem.OPT_SIZE_PLANS, 0)
        s1 = engine.size_stalls
        C = engine.spgemm(A, B)
        assert engine.size_stalls - s1 == first
        C.free()
    finally:
        engine.set_option(pem.OPT_SIZE_PLANS, 1)
        engine.set_option(pem.OPT_STEP1_PATH, 0)
    A.free()
    if B is not A:
        B.free()


@pytest.mark.parametrize("k", [1, 2, 3, 4, 5])
@pytest.mark.parametrize("step1_path", [0, 1, 2])
def test_product_graphs_replay_bit_identical(engine, k, step1_path):
    """PEM_OPT_GRAPHS: the second product of an operand pair is captured as one CUDA graph, later ones are single graph
    launches over the graph's own buffers.  Same bits as the ordinary path; a product called while the previous result
    is alive takes the ordinary path; results of panels, option changes and operand frees keep working."""
    name, tb, (rows, cols, I, J, V) = synth.config(k, small=True)
    A = engine.convert_coo(rows, cols, I, J, V)
    B = engine.convert_coo(rows, cols, I, J, V, transpose=tb)
    _, _, oC = host.spgemm_from_coo(rows, cols, I, J, V, tb)
    engine.set_option(pem.OPT_STEP1_PATH, step1_path)
    engine.set_option(pem.OPT_SIZE_PLANS, 1)
    engine.set_option(pem.OPT_GRAPHS, 1)
    try:
        C = engine.spgemm(A, B)                       # records the sizes
        ref = C.checksum()
        C.free()
        g0 = engine.graph_replays
        l0 = engine.launch_count
        C = engine.spgemm(A, B)                       # captured + launched
        assert engine.graph_replays == g0 + 1, "the second product of a plan should have been captured as a graph"
        per_product = engine.launch_count - l0
        assert per_product > 0
        _assert_same_C(C, oC)
        C.free()
        for _ in range(3):                            # graph launches
            s1, g1, l1 = engine.size_stalls, engine.graph_replays, engine.launch_count
            t = pem.Times()
            C = engine.spgemm(A, B, times=t)
            assert engine.graph_replays == g1 + 1 and engine.size_stalls == s1
            assert engine.launch_count - l1 == per_product
            assert C.checksum() == ref
            assert t.step1_ms > 0 and t.step3_ms >= 0 and t.kernel_ms > 0      # the timing events live inside the graph
            _assert_same_C(C, oC)
            C.free()
        # previous result alive: the graph's buffers are lent out, so this product runs the ordinary way
        C1 = engine.spgemm(A, B)
        g1 = engine.graph_replays
        C2 = engine.spgemm(A, B)
        assert engine.graph_replays == g1
        _assert_same_C(C1, oC); _assert_same_C(C2, oC)
        assert C1.array("row_col_idx").size == oC.nnz           # an array added to a graph-backed result later on
        C1.free(); C2.free()
        C = engine.spgemm(A, B)                       # lent buffers are back: a graph launch again
        assert engine.graph_replays == g1 + 1
        _assert_same_C(C, oC)
        C.free()
        # panels have their own plans and graphs
        bounds = engine.partition_panels(A, B, 2)
        for rep in range(3):
            g1 = engine.graph_replays
            parts = [engine.spgemm(A, B, panel=(int(bounds[i]), int(bounds[i + 1]))) for i in range(2)]
            assert engine.graph_replays - g1 == (0 if rep == 0 else 2)
            assert sum(p.info.nnz for p in parts) == oC.nnz
            coo = [p_.to_coo() for p_ in parts]
            ro, co, vo = oC.to_coo()
            for j, want in enumerate((ro, co, vo)):
                assert np.array_equal(np.concatenate([x[j] for x in coo]), want)
            for p_ in parts:
                p_.free()
        # another kernel choice is not what the graph holds: ordinary path, same bits
        engine.set_option(pem.OPT_OWNER, 2)
        g1 = engine.graph_replays
        C = engine.spgemm(A, B)
        assert engine.graph_replays == g1
        _assert_same_C(C, oC)
        C.free()
        engine.set_option(pem.OPT_OWNER, 0)
        # a budget of zero: nothing is captured
        engine.set_option(pem.OPT_GRAPHS, 1)          # drops the graphs
        engine.set_option(pem.OPT_GRAPH_LIMIT_MB, 0)
        for rep in range(3):
            g1 = engine.graph_replays
            C = engine.spgemm(A, B)
            assert engine.graph_replays == g1
            _assert_same_C(C, oC)
            C.free()
        engine.set_option(pem.OPT_GRAPH_LIMIT_MB, 16384)
        engine.set_option(pem.OPT_GRAPHS, 1)
        engine.set_option(pem.OPT_GRAPHS, 0)
        g1 = engine.graph_replays
        C = engine.spgemm(A, B)
        assert engine.graph_replays == g1
        _assert_same_C(C, oC)
        C.free()
        # freeing an operand drops its graphs; the buffers are reusable by whatever comes next
        engine.set_option(pem.OPT_GRAPHS, 1)
        for _ in range(3):
            C = engine.spgemm(A, B); C.free()
        C = engine.spgemm(A, B)                       # graph-backed and alive while the operands go away
    finally:
        engine.set_option(pem.OPT_GRAPHS, 1)
        engine.set_option(pem.OPT_GRAPH_LIMIT_MB, 16384)
        engine.set_option(pem.OPT_OWNER, 0)
        engine.set_option(pem.OPT_STEP1_PATH, 0)
    if B is not A:
        B.free()
    A.free()
    _assert_same_C(C, oC)                             # the result outlives its graph's plan
    C.free()
    A = engine.convert_coo(rows, cols, I, J, V)
    B = engine.convert_coo(rows, cols, I, J, V, transpose=tb)
    for _ in range(3):
        C = engine.spgemm(A, B)
        _assert_same_C(C, oC)
        C.free()
    B.free(); A.free()


@pytest.mark.parametrize("k", [1, 4, 2])
def test_abandoned_graph_capture_falls_back(engine, k):
    """A capture that cannot complete is given up and the product redone the ordinary way: here the recording product
    ran the row-owner kernels (no step-3 views on the operands), so the capture of the next product would have to build
    the operands' views out of a graph arena, which the engine refuses."""
    name, tb, (rows, cols, I, J, V) = synth.config(k, small=True)
    A = engine.convert_coo(rows, cols, I, J, V)
    B = engine.convert_coo(rows, cols, I, J, V, transpose=tb)
    _, _, oC = host.spgemm_from_coo(rows, cols, I, J, V, tb)
    engine.set_option(pem.OPT_GRAPHS, 1)
    engine.set_option(pem.OPT_OWNER, 1)
    try:
        C = engine.spgemm(A, B)
        _assert_same_C(C, oC)
        C.free()
        engine.set_option(pem.OPT_OWNER, 0)
        l0 = engine.launch_count
        C = engine.spgemm(A, B)                       # ordinary path with the default kernels, after the abandoned capture
        per_product = engine.launch_count - l0
        for rep in range(3):
            g1, s1, l1 = engine.graph_replays, engine.size_stalls, engine.launch_count
            _assert_same_C(C, oC)
            C.free()
            C = engine.spgemm(A, B)
            assert engine.graph_replays == g1 and engine.size_stalls == s1      # no graph for this plan, sizes still replayed
            assert engine.launch_count - l1 <= per_product                        # (the first one also built the views)
        _assert_same_C(C, oC)
        C.free()
    finally:
        engine.set_option(pem.OPT_OWNER, 0)
    B.free(); A.free()


@pytest.mark.parametrize("owner", [1, 2, 3, 4])
@pytest.mark.parametrize("k", [1, 2, 3, 4])
def test_owner_variants_are_bit_identical(engine, k, owner):
    """PEM_OPT_OWNER = 1 (row-owner), 2 (entry-owner), 3 (tile-class kernel) must give the same bits as
    the automatic choice and as the oracle."""
    name, tb, (rows, cols, I, J, V) = synth.config(k, small=True)
    A = engine.convert_coo(rows, cols, I, J, V)
    B = engine.convert_coo(rows, cols, I, J, V, transpose=tb)
    C0 = engine.spgemm(A, B)
    engine.set_option(pem.OPT_OWNER, owner)
    try:
        C1 = engine.spgemm(A, B)
    finally:
        engine.set_option(pem.OPT_OWNER, 0)
    assert np.array_equal(C0.array("masks"), C1.array("masks"))
    assert np.array_equal(C0.array("tile_nnz_ptr"), C1.array("tile_nnz_ptr"))
    assert np.array_equal(C0.array("vals"), C1.array("vals"))
    assert np.array_equal(C0.array("row_col_idx"), C1.array("row_col_idx"))
    _, _, oC = host.spgemm_from_coo(rows, cols, I, J, V, tb)
    _assert_same_C(C1, oC)
    C0.free(); C1.free(); A.free(); B.free()


@pytest.mark.parametrize("kernel", [1, 2, 3])
@pytest.mark.parametrize("keep_empty", [0, 1])
@pytest.mark.parametrize("k", [1, 2, 3, 4, 5])
def test_step2_kernels_match_tile_oracle(engine, k, keep_empty, kernel):
    """The step-2 mask kernels (lane per pair in list form and in row-mask form; sixteen lanes per C' tile) against the numpy restatement of
    compute_CMasksAndOffsets (spgemm.cu:499-550), and the values that step 3 derives from their hit blocks."""
    name, tb, (rows, cols, I, J, V) = synth.config(k, small=True)
    engine.set_option(pem.OPT_KEEP_EMPTY_TILES, keep_empty)
    engine.set_option(pem.OPT_STEP2_KERNEL, kernel)
    try:
        A = engine.convert_coo(rows, cols, I, J, V)
        B = engine.transpose(A) if tb else A
        OA = tiles.tile_format(rows, cols, I, J, V)
        OB = tiles.tile_format(rows, cols, I, J, V, transpose=tb)
        P = tiles.tiled_product(OA, OB, keep_empty=bool(keep_empty))
        C = engine.step1(A, B)
        engine.step2(A, B, C)
        assert np.array_equal(C.array("masks").reshape(-1, 16), P.c_masks)
        assert np.array_equal(C.array("tile_nnz_ptr"), P.c_tile_nnz_ptr)
        engine.step3(A, B, C)
        _, _, Co = host.spgemm_from_coo(rows, cols, I, J, V, tb)
        _assert_same_C(C, Co)
        C.free()
        if B is not A:
            B.free()
        A.free()
    finally:
        engine.set_option(pem.OPT_KEEP_EMPTY_TILES, 0)
        engine.set_option(pem.OPT_STEP2_KERNEL, 0)


@pytest.mark.parametrize("small_e,small_np", [(0, 0), (256, 1 << 20), (256, 1), (2, 4), (8, 0)])
@pytest.mark.parametrize("k", [1, 2, 3, 4, 5])
def test_step3_tile_classes_are_bit_identical(engine, k, small_e, small_np):
    """The tile-class kernel of step 3 with its thresholds pushed to the extremes, so that every tile goes
    through the warp mappings (staged records / hit blocks), or every tile through the one-thread mapping
    (single-pair walk / hit blocks): same bits as the oracle whatever the class."""
    name, tb, (rows, cols, I, J, V) = synth.config(k, small=True)
    A = engine.convert_coo(rows, cols, I, J, V)
    B = engine.transpose(A) if tb else A
    _, _, oC = host.spgemm_from_coo(rows, cols, I, J, V, tb)
    engine.set_option(pem.OPT_S3_SMALL_NNZ, small_e)
    engine.set_option(pem.OPT_S3_SMALL_PAIRS, small_np)
    engine.set_option(pem.OPT_OWNER, 3)
    try:
        for keep in (0, 1):
            engine.set_option(pem.OPT_KEEP_EMPTY_TILES, keep)
            C = engine.spgemm(A, B)
            _assert_same_C(C, oC)
            C.free()
    finally:
        engine.set_option(pem.OPT_KEEP_EMPTY_TILES, 0)
        engine.set_option(pem.OPT_OWNER, 0)
        engine.set_option(pem.OPT_S3_SMALL_NNZ, 8)
        engine.set_option(pem.OPT_S3_SMALL_PAIRS, 64)
    if B is not A:
        B.free()
    A.free()


@pytest.mark.parametrize("k", [2, 3])
def test_step1_hash_rows_agree_at_full_size(engine, k):
    """PEM_OPT_STEP1_PATH = 5 (hash accumulators on every tile row of at most 1024 products, bitmap on the hub
    rows) against expand-sort-compress at BASELINE.json sizes: identical C' structure, pair lists and value bits."""
    name, tb, (rows, cols, I, J, V) = synth.config(k)
    A = engine.convert_coo(rows, cols, I, J, V)
    B = engine.convert_coo(rows, cols, I, J, V, transpose=True) if tb else A
    engine.set_option(pem.OPT_STEP1_PATH, 2)
    try:
        C0 = engine.spgemm(A, B)
        engine.set_option(pem.OPT_STEP1_PATH, 5)
        C1 = engine.spgemm(A, B)
    finally:
        engine.set_option(pem.OPT_STEP1_PATH, 0)
    assert (C0.info.tiles, C0.info.pairs, C0.info.nnz) == (C1.info.tiles, C1.info.pairs, C1.info.nnz)
    for name in ("row_ptr", "tile_row", "tile_col", "pair_ptr", "pairs_a", "pairs_b", "tile_nnz_ptr", "vals"):
        assert np.array_equal(C0.array(name), C1.array(name)), name
    C0.free(); C1.free()
    if B is not A:
        B.free()
    A.free()


@pytest.mark.parametrize("esc", [3, 4])
@pytest.mark.parametrize("k", [2, 3])
def test_step1_paths_agree_at_full_size(engine, k, esc):
    """BASELINE.json sizes (too big for the numpy tile oracle): the two step-1 algorithms must
    produce identical C' structure and pair lists, and step 3 identical value bits."""
    name, tb, (rows, cols, I, J, V) = synth.config(k)
    A = engine.convert_coo(rows, cols, I, J, V)
    B = engine.convert_coo(rows, cols, I, J, V, transpose=True) if tb else A
    engine.set_option(pem.OPT_STEP1_PATH, esc)
    try:
        C0 = engine.spgemm(A, B)
        engine.set_option(pem.OPT_STEP1_PATH, 1)
        C1 = engine.spgemm(A, B)
    finally:
        engine.set_option(pem.OPT_STEP1_PATH, 0)
    assert (C0.info.tiles, C0.info.pairs, C0.info.nnz) == (C1.info.tiles, C1.info.pairs, C1.info.nnz)
    for name in ("row_ptr", "tile_row", "tile_col", "pair_ptr", "pairs_a", "pairs_b", "tile_nnz_ptr", "vals"):
        assert np.array_equal(C0.array(name), C1.array(name)), name
    C0.free(); C1.free()
    if B is not A:
        B.free()
    A.free()


def test_wide_index_space_uses_64bit_sort_keys(engine):
    """16.7M x 16.7M with the nonzeros on ~3000 scattered rows/columns: ~1M tile rows and a tile-column
    window of ~1M need 40 key bits, i.e. the 64-bit-key instantiation of expand-sort-compress."""
    rng = np.random.default_rng(7)
    n = 1 << 24
    ids = np.sort(rng.choice(n, size=3000, replace=False)).astype(np.int64)
    I = ids[rng.integers(0, ids.size, 120_000)]
    J = ids[rng.integers(0, ids.size, 120_000)]
    key = np.unique(I * n + J)
    I = (key // n).astype(np.int32); J = (key % n).astype(np.int32)
    V = rng.uniform(-1, 1, I.size)
    _, _, oC = host.spgemm_from_coo(n, n, I, J, V, False)
    A = engine.convert_coo(n, n, I, J, V)
    for path in (3, 4):
        engine.set_option(pem.OPT_STEP1_PATH, path)
        try:
            C = engine.spgemm(A, A)
        finally:
            engine.set_option(pem.OPT_STEP1_PATH, 0)
        _assert_same_C(C, oC)
        C.free()
    A.free()


@pytest.mark.parametrize("k", [2, 4])
def test_esc_count_then_write_variant(engine, k):
    """The variant of expand-sort-compress used when product-sized staging buffers would not fit
    (count per chunk, scan, write exactly): same arrays as the staged variant; with and without the
    block-local row sort (PEM_OPT_ESC_VARIANT bits)."""
    name, tb, (rows, cols, I, J, V) = synth.config(k, small=True)
    A = engine.convert_coo(rows, cols, I, J, V)
    got = {}
    try:
        for variant in (0, 1, 2, 3):
            engine.set_option(pem.OPT_ESC_VARIANT, variant)
            for path in (3, 4):
                engine.set_option(pem.OPT_STEP1_PATH, path)
                C = engine.spgemm(A, A)
                got[(variant, path)] = [C.array(x) for x in ("row_ptr", "tile_col", "pair_ptr", "pairs_a", "pairs_b", "vals")]
                C.free()
    finally:
        engine.set_option(pem.OPT_ESC_VARIANT, 0)
        engine.set_option(pem.OPT_STEP1_PATH, 0)
    ref = got[(0, 3)]
    for key, arrs in got.items():
        for a, b in zip(ref, arrs):
            assert np.array_equal(a, b), key
    pool = engine.pool_bytes
    A.free()
    engine.trim()                               # cached blocks go back to the driver
    assert engine.pool_bytes <= pool


def test_config2_full_size_matches_oracle(engine):
    """BASELINE config 2 at full size (3.09 M nonzeros, nnz(C) = 67.7 M): structure and values of C
    against the host oracle, bit for bit."""
    name, tb, (rows, cols, I, J, V) = synth.config(2)
    A = engine.convert_coo(rows, cols, I, J, V)
    C = engine.spgemm(A, A)
    oA, oB, oC = host.spgemm_from_coo(rows, cols, I, J, V, False)
    assert engine.count_flop(A, A) == host.flop(oA, oB) == 92_217_721
    assert C.info.nnz == oC.nnz == 67_736_942
    _assert_same_C(C, oC)
    C.free(); A.free()


def _assert_same_C_lowmem(Cres, oC, row0=0):
    """_assert_same_C for results of hundreds of millions of entries: array by array, without building
    the oracle's row array (rows are compared through per-row counts)."""
    r, c, v = Cres.to_coo()
    assert r.size == oC.nnz
    assert np.array_equal(c, oC.idx)                                   # structure: bit-exact
    cnt = np.bincount(r - row0, minlength=oC.rows) if r.size else np.zeros(oC.rows, np.int64)
    assert cnt.size == oC.rows and np.array_equal(cnt, np.diff(oC.ptr))
    assert r.size == 0 or bool(np.all(np.diff(r) >= 0))
    del r, c
    _assert_bits(v, oC.val)                                            # same fma order => same bits (tolerance 1e-12 is implied)


def test_config3_full_size_matches_oracle(engine):
    """BASELINE config 3 at full size (A*A^T, 9.94 M nonzeros, nnz(C) = 81.6 M): structure and values of C
    against the host oracle, bit for bit."""
    name, tb, (rows, cols, I, J, V) = synth.config(3)
    A = engine.convert_coo(rows, cols, I, J, V)
    B = engine.transpose(A)
    C = engine.spgemm(A, B)
    oA, oB, oC = host.spgemm_from_coo(rows, cols, I, J, V, True)
    assert engine.count_flop(A, B) == host.flop(oA, oB)
    assert C.info.nnz == oC.nnz
    _assert_same_C_lowmem(C, oC)
    C.free(); B.free(); A.free()


def test_config4_full_size_matches_oracle(engine):
    """BASELINE config 4 at full size (96.9 M nonzeros, nnz(C) = 470 M): every column index and every value
    bit of C against the host oracle (about 16 GB of host memory for the two COO copies)."""
    name, tb, (rows, cols, I, J, V) = synth.config(4)
    A = engine.convert_coo(rows, cols, I, J, V)
    C = engine.spgemm(A, A)
    oA, oB, oC = host.spgemm_from_coo(rows, cols, I, J, V, False)
    del I, J, V
    assert C.info.nnz == oC.nnz == 470_380_286
    _assert_same_C_lowmem(C, oC)
    C.free(); A.free()


def test_config5_full_size_matches_oracle_panel_by_panel(engine):
    """BASELINE config 5 at full size (R-MAT scale 22, 67.1 M nonzeros, nnz(C) = 2.5 G > 2^31): C does not fit
    one GPU in tiled form, so it is produced in 16 tile-row panels; each panel is compared with the host
    oracle run on the matching row slice of A (host memory stays bounded by one panel)."""
    name, tb, (rows, cols, I, J, V) = synth.config(5)
    A = engine.convert_coo(rows, cols, I, J, V)
    oA = host.coo_to_csr(rows, cols, I, J, V)
    del I, J, V
    assert engine.count_flop(A, A) == host.flop(oA, oA)
    nparts = 16
    bounds = engine.partition_panels(A, A, nparts)
    total = 0
    for p in range(nparts):
        rb, re = int(bounds[p]), int(bounds[p + 1])
        C = engine.spgemm(A, A, panel=(rb, re))
        oC = host.spgemm(host.row_slice(oA, 16 * rb, 16 * re), oA)
        _assert_same_C_lowmem(C, oC, row0=16 * rb)
        total += oC.nnz
        C.free()
        del oC
    assert total > 2**31                    # the reference's int32 C_nnz cannot hold it (SURVEY.md section 4 quirk 6)
    A.free()


def test_config4_full_size_known_answers_and_checksum(engine):
    """BASELINE config 4 at full size against the analytic figures pinned in SURVEY.md section 8c and a
    size-independent property: sum(C) = sum_k colsum_k(A) * rowsum_k(A)."""
    name, tb, (rows, cols, I, J, V) = synth.config(4)
    assert (rows, I.size) == (5_147_788, 96_915_634)
    A = engine.convert_coo(rows, cols, I, J, V)
    assert A.info.tiles == 5_418_031
    assert engine.count_flop(A, A) == 1_828_978_714
    engine.set_option(pem.OPT_KEEP_EMPTY_TILES, 1)          # the reference's C' (structurally reachable tiles)
    try:
        C = engine.step1(A, A)
        assert (C.info.tiles, C.info.pairs) == (23_814_841, 91_431_915)
        C.free()
    finally:
        engine.set_option(pem.OPT_KEEP_EMPTY_TILES, 0)
    C = engine.spgemm(A, A)
    assert C.info.nnz == 470_380_286
    s, a = C.checksum()
    rowsum = np.bincount(I, weights=V, minlength=rows)
    colsum = np.bincount(J, weights=V, minlength=cols)
    want = float(np.dot(colsum, rowsum))
    assert abs(s - want) <= 1e-9 * abs(want) and abs(a - want) <= 1e-9 * abs(want)   # all values positive
    C.free(); A.free()


def test_fuzz_all_variants_against_oracle(engine):
    """Seeded sweep over shapes, densities, products and every algorithm variant: step-1 path
    (bitmap, tile-level / row-sliced expand-sort-compress), step-3 mapping (four kernels), reference-
    faithful empty tiles on/off, tile-row panels.  Structure and value bits against the host oracle."""
    rng = np.random.default_rng(2026)
    for case in range(36):
        m = int(rng.choice([1, 7, 16, 33, 100, 257, 900]))
        aat = bool(rng.integers(0, 2))
        n = int(rng.choice([1, 5, 16, 48, 130, 700, 3000])) if aat else m
        nnz = int(min(m * n, rng.choice([1, 3, 40, 400, 3000, 12000])))
        rows, cols, I, J, V = synth.random_sparse(m, n, nnz, seed=1000 + case, integer_values=bool(case % 3 == 0))
        if case % 5 == 0 and I.size:                      # a dense block somewhere: full tiles, long pair lists
            k = min(m, n, 20)
            bi, bj = np.divmod(np.arange(k * k, dtype=np.int32), k)
            key = np.unique(np.concatenate([I.astype(np.int64) * n + J, bi.astype(np.int64) * n + bj]))
            I = (key // n).astype(np.int32); J = (key % n).astype(np.int32)
            V = rng.uniform(-1, 1, I.size)
        _, _, oC = host.spgemm_from_coo(rows, cols, I, J, V, aat)
        ro, co, vo = oC.to_coo()
        A = engine.convert_coo(rows, cols, I, J, V)
        B = engine.transpose(A) if aat else A
        path = (1, 3, 4, 5)[case % 4]
        owner = (2, 0, 1, 3, 4)[case % 5]
        keep = case % 2
        engine.set_option(pem.OPT_STEP2_KERNEL, (1, 2, 0, 3)[case % 4])
        engine.set_option(pem.OPT_STEP1_PATH, path)
        engine.set_option(pem.OPT_OWNER, owner)
        engine.set_option(pem.OPT_KEEP_EMPTY_TILES, keep)
        try:
            nparts = 1 + case % 3
            bounds = engine.partition_panels(A, B, nparts)
            parts = []
            for p in range(nparts):
                C = engine.spgemm(A, B, panel=(bounds[p], bounds[p + 1]))
                parts.append(C.to_coo())
                C.free()
        finally:
            engine.set_option(pem.OPT_STEP1_PATH, 0)
            engine.set_option(pem.OPT_OWNER, 0)
            engine.set_option(pem.OPT_KEEP_EMPTY_TILES, 0)
            engine.set_option(pem.OPT_STEP2_KERNEL, 0)
        r = np.concatenate([x[0] for x in parts]); c = np.concatenate([x[1] for x in parts])
        v = np.concatenate([x[2] for x in parts])
        tag = f"case {case}: {m}x{n} nnz {I.size} aat {aat} path {path} owner {owner} keep {keep} parts {nparts}"
        assert np.array_equal(r, ro) and np.array_equal(c, co), tag
        _assert_bits(v, vo, tag)
        if B is not A:
            B.free()
        A.free()
