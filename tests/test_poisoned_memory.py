"""Every path against poisoned device memory.  The engine's allocator recycles freed blocks by size, so a repeated
product usually gets its own earlier blocks back, still holding that product's results, and a first allocation
takes pool memory that is probably zero.  Under either, a kernel that reads memory nothing wrote (a missing memset,
an element a scan never writes, a hit word past the last pair) can still produce the right answer.

PEM_OPT_POISON fills every block the allocator hands out with one byte.  Each pattern gets a context of its own,
set before the first conversion, so operands and their lazily built caches (row slices, step-3 views) are poisoned
too:
  0x00  what fresh memory probably looks like
  0xFF  NaN doubles, index -1, full masks
  0x5A  plausible masks and large positive integers
Every array the engine exposes is compared with the oracle bit for bit where one exists.  Across the three
patterns every array, the result info (tile products included), the path indicators, the panel bounds and the
checksum must be identical: the engine's reductions are deterministic, so any difference is a read of memory that
nothing wrote."""
import ctypes

import numpy as np
import pytest

import pem_spgemm_b200 as pem
import test_error_paths as error_paths
from oracle import host, tiles
from pem_spgemm_b200 import synth
from test_general_product import DENSITY, SHAPES, Opts, _assert_bits, _rand_tiled
from test_gpu_parity import _check_tiled

pytestmark = pytest.mark.gpu

PATTERNS = [0x00, 0xFF, 0x5A]


@pytest.fixture(scope="module", params=PATTERNS, ids=[f"0x{p:02X}" for p in PATTERNS])
def pctx(request):
    ctx = pem.Context(0)
    ctx.set_option(pem.OPT_POISON, 0x100 | request.param)
    yield ctx, request.param
    ctx.close()


# ---------------------------------------------------------------------------------------------------------------
# inputs
# ---------------------------------------------------------------------------------------------------------------
def _t(X):
    rows, cols, I, J, V = X
    return cols, rows, J.copy(), I.copy(), V.copy()


def _rect(shape, da, db):
    """The independent rectangular operands of test_general_product_every_variant."""
    m, k, n, ta, tb = SHAPES[shape]
    rng = np.random.default_rng(sum(map(ord, shape + da + db)))
    return _rand_tiled(m, k, ta, DENSITY[da], rng), _rand_tiled(k, n, tb, DENSITY[db], rng)


def _config(k):
    _, tb, A = synth.config(k, small=True)
    return A, (_t(A) if tb else None)


def _empty_product():
    """A (40 x 40, columns 0-3 only) times B (rows 5-9 and 20-39 only): C is empty, but A's tiles in tile column 0
    meet B's tiles in tile row 0, so C' has reachable tiles with empty masks under keep-empty."""
    I = np.arange(0, 40, 3).repeat(4).astype(np.int32)
    J = np.tile(np.arange(4), I.size // 4).astype(np.int32)
    r = np.concatenate([np.arange(5, 10), np.arange(20, 40)]).astype(np.int32)
    c = (r * 7 % 40).astype(np.int32)
    return (40, 40, I, J, 1.0 + np.arange(I.size) / 8), (40, 40, r, c, -0.5 - np.arange(r.size) / 4)


def _cases():
    """name -> (A, B or None for A*A, conversion path)"""
    z = np.zeros(0, np.int32)
    c = {}
    for k, conv in zip(range(1, 6), ("host_coo", "device_coo", "device_transpose", "csr_host", "async")):
        A, B = _config(k)
        c[f"config{k}"] = (A, B, conv)
    c["hyper_x_dense"] = (*_rect("wide", "hyper", "dense"), "fp32")
    c["dense_x_hyper"] = (*_rect("tall", "dense", "hyper"), "device_coo")
    L = synth.random_sparse(48, 6000, 40000, seed=21)      # test_dense_tiles_with_long_pair_lists: 375 pairs per C' tile
    c["long_pair_lists"] = (L, _t(L), "device_transpose")
    c["empty_operand"] = ((40, 40, z, z.copy(), np.zeros(0)), None, "host_coo")
    c["one_by_one"] = ((1, 1, np.zeros(1, np.int32), np.zeros(1, np.int32), np.array([-2.5])), None, "csr_host")
    c["empty_product"] = (*_empty_product(), "fp32")
    return c


CASES = _cases()
_ORACLES = {}


class _Oracle:
    def __init__(self, name):
        A, B, conv = CASES[name]
        B = B if B is not None else A
        f32 = conv == "fp32"
        cast = (lambda X: (*X[:4], X[4].astype(np.float32).astype(np.float64))) if f32 else (lambda X: X)
        self.oA, self.oB = host.coo_to_csr(*cast(A)), host.coo_to_csr(*cast(B))
        self.C = (host.spgemm_f32 if f32 else host.spgemm)(self.oA, self.oB)
        self.flop = host.flop(self.oA, self.oB)
        self.TA, self.TB = TA, TB = tiles.tile_format(*cast(A)), tiles.tile_format(*cast(B))
        self.tile_rows = TA.tile_rows
        self.P = {keep: tiles.tiled_product(TA, TB, keep_empty=bool(keep)) for keep in (0, 1)}
        self.rci = {}

    def row_col_idx(self, keep):
        """(r << 4) | c of every set mask bit, tile by tile, row-major"""
        if keep not in self.rci:
            m = self.P[keep].c_masks
            t, r = np.nonzero(m)
            bits = (m[t, r].astype(np.int64)[:, None] >> np.arange(16)) & 1
            idx, cc = np.nonzero(bits)
            self.rci[keep] = ((r[idx] << 4) | cc).astype(np.uint8)
        return self.rci[keep]

    def panel(self, rb, re):
        """rows, cols, vals and the CSR row pointer (from 0) of C's rows in tile rows [rb, re)"""
        oC = self.C
        r0, r1 = min(oC.rows, 16 * rb), min(oC.rows, 16 * re)
        b, e = int(oC.ptr[r0]), int(oC.ptr[r1])
        r, c, v = oC.to_coo()
        return r[b:e], c[b:e], v[b:e], oC.ptr[r0:r1 + 1] - b


def _oracle(name):
    if name not in _ORACLES:
        _ORACLES[name] = _Oracle(name)
    return _ORACLES[name]


def _convert(ctx, name, keep_alive):
    """(A, B) handles of a case through its conversion path; B is A for A*A."""
    A, B, conv = CASES[name]

    def one(X):
        rows, cols, I, J, V = X
        if conv == "device_coo":
            import torch
            d = [torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (I, J, V)]
            torch.cuda.synchronize()
            keep_alive.extend(d)
            return ctx.convert_coo(rows, cols, *(t.data_ptr() for t in d), nnz=I.size)
        if conv == "csr_host":
            o = host.coo_to_csr(*X)
            return ctx.convert_csr(rows, cols, o.ptr.astype(np.int32), o.idx, o.val)
        if conv == "async":
            import torch
            h = [torch.from_numpy(np.ascontiguousarray(x)).pin_memory() for x in (I, J, V)]
            keep_alive.extend(h)                  # the upload may still read V after the call returns
            ctx.set_option(pem.OPT_ASYNC_VALUES, 1)
            try:
                return ctx.convert_coo(rows, cols, *(t.numpy() for t in h))
            finally:
                ctx.set_option(pem.OPT_ASYNC_VALUES, 0)
        return ctx.convert_coo(*X, dtype=np.float32 if conv == "fp32" else np.float64)

    tA = one(A)
    if B is None:
        return tA, tA
    if conv == "device_transpose":
        Bt = ctx.convert_coo(*_t(B))
        try:
            return tA, ctx.transpose(Bt)
        finally:
            Bt.free()
    return tA, one(B)


def _free(tA, tB):
    if tB is not tA:
        tB.free()
    tA.free()


# ---------------------------------------------------------------------------------------------------------------
# what a result exposes, and its comparison across patterns
# ---------------------------------------------------------------------------------------------------------------
R_NAMES = ("row_ptr", "tile_row", "tile_col", "pair_ptr", "pairs_a", "pairs_b", "masks", "tile_nnz_ptr",
           "row_col_idx", "vals")


def _fingerprint(ctx, C):
    i = C.info
    fp = {n: C.array(n) for n in R_NAMES}
    fp["info"] = np.array([i.tile_row_begin, i.tile_row_end, i.rows, i.cols, i.tiles, i.pairs, i.nnz,
                           i.tile_products], np.int64)
    fp["coo_rows"], fp["coo_cols"], fp["coo_vals"] = C.to_coo()
    if C.dtype == np.float64:
        fp["csr_ptr"], fp["csr_cols"], fp["csr_vals"] = C.to_csr()
    fp["checksum"] = np.array(C.checksum())
    return fp


_SEEN = {}


def _same_across_patterns(pattern, key, fp):
    """The first pattern to run a key records what it saw; every other pattern must see the same bytes."""
    if key not in _SEEN or _SEEN[key][0] == pattern:
        _SEEN[key] = (pattern, fp)
        return
    p0, fp0 = _SEEN[key]
    assert fp.keys() == fp0.keys(), key
    for k in fp:
        a, b = np.asarray(fp[k]), np.asarray(fp0[k])
        assert a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes(), \
            f"{key} {k}: differs between poison 0x{p0:02X} and 0x{pattern:02X}"


def _assert_full_result(fp, orc, keep, tag):
    """A result of all of A's tile rows against the tile oracle and the host oracle."""
    P = orc.P[keep]
    for name, want in (("row_ptr", P.c_row_ptr), ("tile_row", P.c_tile_row), ("tile_col", P.c_tile_col),
                       ("pair_ptr", P.pair_ptr), ("pairs_a", P.pairs_a), ("pairs_b", P.pairs_b),
                       ("tile_nnz_ptr", P.c_tile_nnz_ptr)):
        assert np.array_equal(fp[name], want), (tag, name)
    assert np.array_equal(fp["masks"].reshape(-1, 16), P.c_masks), tag
    assert np.array_equal(fp["row_col_idx"], orc.row_col_idx(keep)), tag
    _assert_panel(fp, orc, 0, orc.tile_rows, tag)


def _assert_panel(fp, orc, rb, re, tag):
    r, c, v, rp = orc.panel(rb, re)
    assert np.array_equal(fp["coo_rows"], r) and np.array_equal(fp["coo_cols"], c), tag
    _assert_bits(fp["coo_vals"], v, tag)
    if "csr_ptr" in fp:
        assert np.array_equal(fp["csr_ptr"], rp) and np.array_equal(fp["csr_cols"], c), tag
        _assert_bits(fp["csr_vals"], v, tag)


# ---------------------------------------------------------------------------------------------------------------
# a. every path and variant
# ---------------------------------------------------------------------------------------------------------------
def _variants(ci, f32):
    """Six runs per case, one per step-1 path; the other factors cycle with the case index, so that over the eleven
    cases every ESC variant, keep-empty setting, step-2 kernel, owner and run mode (staged steps, pem_spgemm, three
    panels) meets every pattern.  fp32 runs owners 0, 2 and 4 only."""
    for i in range(6):
        x = i + ci
        owner = x % 5
        if f32:
            owner = {1: 0, 3: 4}.get(owner, owner)
        yield dict(step1_path=i, esc_variant=x % 4, keep_empty_tiles=x % 2, step2_kernel=(i + 2 * ci) % 4,
                   owner=owner), ("staged", "spgemm", "panels")[x % 3]


@pytest.mark.parametrize("name", list(CASES))
def test_every_path_under_poison(pctx, name):
    ctx, pattern = pctx
    ci = list(CASES).index(name)
    orc = _oracle(name)
    keep_alive = []
    tA, tB = _convert(ctx, name, keep_alive)
    f32 = tA.dtype == np.float32
    try:
        assert ctx.count_flop(tA, tB) == orc.flop
        bounds = ctx.partition_panels(tA, tB, 3)
        assert bounds[0] == 0 and bounds[-1] == orc.tile_rows and np.all(np.diff(bounds) >= 0)
        _same_across_patterns(pattern, (name, "bounds"), {"bounds": bounds})
        for vi, (opts, mode) in enumerate(_variants(ci, f32)):
            if mode == "panels" and orc.tile_rows < 3:
                mode = "spgemm"
            tag = f"{name} poison 0x{pattern:02X} {mode} {opts}"
            keep = opts["keep_empty_tiles"]
            with Opts(ctx, **opts):
                if mode == "panels":
                    for q in range(3):
                        C = ctx.spgemm(tA, tB, panel=(bounds[q], bounds[q + 1]))
                        try:
                            fp = _fingerprint(ctx, C)
                            fp["ran"] = np.array([ctx.last_sort_passes, ctx.last_step3_kernel])
                            _assert_panel(fp, orc, bounds[q], bounds[q + 1], f"{tag} panel {q}")
                            _same_across_patterns(pattern, (name, vi, q), fp)
                        finally:
                            C.free()
                    continue
                if mode == "staged":
                    C = ctx.step1(tA, tB)
                    passes = ctx.last_sort_passes
                    ctx.step2(tA, tB, C)
                    ctx.step3(tA, tB, C)
                else:
                    C = ctx.spgemm(tA, tB)
                    passes = ctx.last_sort_passes
                try:
                    fp = _fingerprint(ctx, C)
                    fp["ran"] = np.array([passes, ctx.last_step3_kernel])
                    assert C.dtype == (np.float32 if f32 else np.float64), tag
                    _assert_full_result(fp, orc, keep, tag)
                    _same_across_patterns(pattern, (name, vi), fp)
                finally:
                    C.free()
        # the operands, after every product read them and built their caches
        _check_tiled(tA, orc.TA)
        if tB is not tA:
            _check_tiled(tB, orc.TB)
    finally:
        _free(tA, tB)


# ---------------------------------------------------------------------------------------------------------------
# b. size plans and graphs: ordinary, captured, graph launch
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,nparts", [("config1", 1), ("config3", 2), ("dense_x_hyper", 3)])
def test_replays_under_poison(pctx, name, nparts):
    """Three products of the same handles per panel: the first records its sizes, the second is captured as a graph
    (whose fill nodes poison its arena) and launched, the third is a graph launch.  All three bit-identical to each
    other and to the oracle."""
    ctx, pattern = pctx
    orc = _oracle(name)
    keep_alive = []
    tA, tB = _convert(ctx, name, keep_alive)
    ctx.set_option(pem.OPT_SIZE_PLANS, 1)
    ctx.set_option(pem.OPT_GRAPHS, 1)
    try:
        bounds = ctx.partition_panels(tA, tB, nparts)
        for q in range(nparts):
            first = None
            for run in range(3):
                g0 = ctx.graph_replays
                C = ctx.spgemm(tA, tB, panel=(bounds[q], bounds[q + 1]))
                try:
                    assert ctx.graph_replays - g0 == (1 if run else 0), (name, q, run)
                    fp = _fingerprint(ctx, C)
                    fp["ran"] = np.array([ctx.last_sort_passes, ctx.last_step3_kernel])
                finally:
                    C.free()
                tag = f"{name} poison 0x{pattern:02X} panel {q} run {run}"
                _assert_panel(fp, orc, bounds[q], bounds[q + 1], tag)
                if first is None:
                    first = fp
                else:
                    for k in fp:
                        assert np.asarray(fp[k]).tobytes() == np.asarray(first[k]).tobytes(), (tag, k)
            _same_across_patterns(pattern, ("replay", name, q), first)
    finally:
        _free(tA, tB)


# ---------------------------------------------------------------------------------------------------------------
# c. a stage refused part-way, then retried
# ---------------------------------------------------------------------------------------------------------------
def test_step2_refusal_and_retry_under_poison(pctx):
    error_paths.test_step2_fp32_refused_under_owner_3_and_1_then_retried(pctx[0])


def test_step3_refusal_and_retry_under_poison(pctx):
    error_paths.test_step3_on_dense_tiles_refused_then_retried(pctx[0])


# ---------------------------------------------------------------------------------------------------------------
# d. option off: the blocks of an earlier, different product
# ---------------------------------------------------------------------------------------------------------------
def _products(ctx, name):
    """Fingerprints of A*B under the default options and under path 3 / owner 2 / step-2 kernel 1."""
    keep_alive = []
    tA, tB = _convert(ctx, name, keep_alive)
    out = []
    try:
        for opts in ({}, dict(step1_path=3, owner=2, step2_kernel=1)):
            with Opts(ctx, **opts):
                C = ctx.spgemm(tA, tB)
                try:
                    fp = _fingerprint(ctx, C)
                    fp["ran"] = np.array([ctx.last_sort_passes, ctx.last_step3_kernel])
                    out.append(fp)
                finally:
                    C.free()
    finally:
        _free(tA, tB)
    return out


@pytest.mark.parametrize("first,second", [("config4", "config2"), ("config2", "config4")])
def test_stale_cached_blocks_without_poison(first, second):
    """A dense product (config 4) then a hypersparse one (config 2) in one context, and the other way round: the
    second product runs on the first one's freed blocks and must equal the same product in a new context."""
    with pem.Context(0) as ctx:
        _products(ctx, first)
        m0 = ctx.pool_mallocs
        got = _products(ctx, second)
        reused = ctx.pool_mallocs - m0
    with pem.Context(0) as ctx:
        want = _products(ctx, second)
        assert reused < ctx.pool_mallocs            # some of the first product's blocks were served again
    orc = _oracle(second)
    for fp, fp0 in zip(got, want):
        _assert_panel(fp, orc, 0, orc.tile_rows, second)
        for k in fp:
            assert np.asarray(fp[k]).tobytes() == np.asarray(fp0[k]).tobytes(), (first, second, k)


# ---------------------------------------------------------------------------------------------------------------
# e. caller buffers: written exactly where the export says, never past
# ---------------------------------------------------------------------------------------------------------------
GUARD = 1024
RAGGED = synth.random_sparse(300, 300, 3000, seed=4)      # 19 tile rows, the last one 12 rows high


def _canary_cases(ctx, A, E):
    """(result, rb, re, oracle panel) for the full C, a middle panel, the last (ragged) panel and an empty C."""
    bounds = ctx.partition_panels(A, A, 3)
    assert 0 < bounds[1] < bounds[2] < bounds[3] == 19
    for rb, re in ((0, 19), (int(bounds[1]), int(bounds[2])), (int(bounds[2]), 19)):
        yield ctx.spgemm(A, A, panel=(rb, re)), rb, re, RAGGED
    yield ctx.spgemm(*E), 0, 3, None


def _want(X, Y, rb, re):
    oC = host.spgemm(host.coo_to_csr(*X), host.coo_to_csr(*Y))
    r0, r1 = min(oC.rows, 16 * rb), min(oC.rows, 16 * re)
    b, e = int(oC.ptr[r0]), int(oC.ptr[r1])
    r, c, v = oC.to_coo()
    rp = np.full(16 * (re - rb) + 1, e - b, np.int64)
    rp[:r1 - r0 + 1] = oC.ptr[r0:r1 + 1] - b
    return r[b:e], c[b:e], v[b:e], rp


def test_device_export_canaries(pctx):
    """pem_result_to_coo_device into torch buffers of nnz + 1024 entries (NaN or -1): the first nnz entries and the
    16 * (panel tile rows) + 1 row-pointer entries equal the oracle, the 1024 guard entries are untouched."""
    import torch
    ctx, pattern = pctx
    EA, EB = _empty_product()
    A = ctx.convert_coo(*RAGGED)
    E = (ctx.convert_coo(*EA), ctx.convert_coo(*EB))
    try:
        for C, rb, re, X in _canary_cases(ctx, A, E):
            try:
                n = C.info.nnz
                nrp = 16 * (re - rb) + 1
                dr = torch.full((n + GUARD,), -1, dtype=torch.int32, device="cuda")
                dc = torch.full((n + GUARD,), -1, dtype=torch.int32, device="cuda")
                dv = torch.full((n + GUARD,), float("nan"), dtype=torch.float64, device="cuda")
                drp = torch.full((nrp + GUARD,), -1, dtype=torch.int64, device="cuda")
                nan_bits = dv[-1:].cpu().numpy().view(np.int64)[0]
                torch.cuda.synchronize()
                C.to_coo_device(dr.data_ptr(), dc.data_ptr(), dv.data_ptr(), drp.data_ptr())
                ctx.sync()
                r, c, v, rp = (t.cpu().numpy() for t in (dr, dc, dv, drp))
                wr, wc, wv, wrp = _want(*((RAGGED, RAGGED) if X is not None else (EA, EB)), rb, re)
                tag = f"poison 0x{pattern:02X} panel {rb}..{re}"
                assert n == wr.size, tag
                assert np.array_equal(r[:n], wr) and np.array_equal(c[:n], wc), tag
                _assert_bits(v[:n], wv, tag)
                assert np.array_equal(rp[:nrp], wrp), tag
                assert np.all(r[n:] == -1) and np.all(c[n:] == -1) and np.all(rp[nrp:] == -1), tag
                assert np.all(v[n:].view(np.int64) == nan_bits), tag
            finally:
                C.free()
    finally:
        A.free(); E[0].free(); E[1].free()


def test_host_export_canaries(pctx):
    """pem_result_to_csr and pem_result_to_coo_f32 into host buffers with 1024 guard entries."""
    ctx, pattern = pctx
    L = pem.load()
    EA, EB = _empty_product()
    A = ctx.convert_coo(*RAGGED)
    E = (ctx.convert_coo(*EA), ctx.convert_coo(*EB))
    try:
        for C, rb, re, X in _canary_cases(ctx, A, E):
            try:
                n = C.info.nnz
                nrows = max(0, min(C.info.rows, 16 * re) - 16 * rb)
                rp = np.full(nrows + 1 + GUARD, -1, np.int64)
                c = np.full(n + GUARD, -1, np.int32)
                v = np.full(n + GUARD, np.nan)
                ctx._check(L.pem_result_to_csr(ctx._h, C._h, pem._ptr(rp), pem._ptr(c), pem._ptr(v)))
                wr, wc, wv, wrp = _want(*((RAGGED, RAGGED) if X is not None else (EA, EB)), rb, re)
                tag = f"poison 0x{pattern:02X} panel {rb}..{re}"
                assert np.array_equal(rp[:nrows + 1], wrp[:nrows + 1]) and np.array_equal(c[:n], wc), tag
                _assert_bits(v[:n], wv, tag)
                assert np.all(rp[nrows + 1:] == -1) and np.all(c[n:] == -1) and np.all(np.isnan(v[n:])), tag
            finally:
                C.free()
    finally:
        A.free(); E[0].free(); E[1].free()
    rows, cols, I, J, V = RAGGED
    A32 = ctx.convert_coo(rows, cols, I, J, V, dtype=np.float32)
    try:
        C = ctx.spgemm(A32, A32)
        try:
            n = C.info.nnz
            r = np.full(n + GUARD, -1, np.int32); c = np.full(n + GUARD, -1, np.int32)
            v = np.full(n + GUARD, np.nan, np.float32)
            ctx._check(L.pem_result_to_coo_f32(ctx._h, C._h, pem._ptr(r), pem._ptr(c), pem._ptr(v)))
            o = host.coo_to_csr(rows, cols, I, J, V.astype(np.float32).astype(np.float64))
            ro, co, vo = host.spgemm_f32(o, o).to_coo()
            assert np.array_equal(r[:n], ro) and np.array_equal(c[:n], co)
            _assert_bits(v[:n], vo)
            assert np.all(r[n:] == -1) and np.all(c[n:] == -1) and np.all(np.isnan(v[n:]))
        finally:
            C.free()
    finally:
        A32.free()


# ---------------------------------------------------------------------------------------------------------------
# f. the option itself
# ---------------------------------------------------------------------------------------------------------------
def test_poison_option_values_and_plans():
    """Only 0 and 0x100 | byte are accepted; setting the option drops the remembered sizes (the next product stalls
    again, so no graph captured without fill nodes runs); with and without it a product launches the same kernels
    and takes the same pool allocations."""
    rows, cols, I, J, V = RAGGED
    with pem.Context(0) as ctx:
        for bad in (-1, 1, 0xFF, 0x5A, 0x200, 0x1000, 1 << 40):
            with pytest.raises(pem.PemError) as e:
                ctx.set_option(pem.OPT_POISON, bad)
            assert e.value.code == -2, bad
        for ok in (0x100, 0x1FF, 0x15A, 0):
            ctx.set_option(pem.OPT_POISON, ok)
        A = ctx.convert_coo(rows, cols, I, J, V)
        for _ in range(3):                          # records, captures, replays
            ctx.spgemm(A, A).free()
        s0 = ctx.size_stalls
        ctx.spgemm(A, A).free()
        assert ctx.size_stalls == s0
        ctx.set_option(pem.OPT_POISON, 0x1A5)
        ctx.spgemm(A, A).free()
        assert ctx.size_stalls > s0
        A.free()
    counts = []
    for value in (0, 0x1FF):
        with pem.Context(0) as ctx:
            ctx.set_option(pem.OPT_POISON, value)
            A = ctx.convert_coo(rows, cols, I, J, V)
            for _ in range(3):
                C = ctx.spgemm(A, A)
                C.to_coo()
                C.free()
            A.free()
            counts.append((ctx.launch_count, ctx.pool_mallocs))
    assert counts[0] == counts[1], counts
