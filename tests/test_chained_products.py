"""Results as operands: Result.to_tiled (pem_result_to_tiled) turns a complete result into a tiled matrix, and
Tiled.refresh_from (pem_tiled_refresh_from_result) writes a recomputed result's values into it in place.

The handle must be, array for array, the one pem_convert_coo builds from the result's COO export, so every test of
the structure compares with that route; chains are compared with the host oracle run twice.  Values are compared bit
for bit (the sign of zero counts, a NaN matches any NaN)."""
import numpy as np
import pytest

import pem_spgemm_b200 as pem
from oracle import host
from pem_spgemm_b200 import synth
from test_general_product import F32, F64, Mat, Opts, _assert_bits, _rand_tiled, pair_family
from test_value_updates import CASES, _assert_result, _operands, _vals, _with

pytestmark = pytest.mark.gpu

ARG = -2
ARRAYS = list(pem.T_ARRAYS)


# ---------------------------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------------------------
def _info(T):
    i = T.info
    return i.rows, i.cols, i.nnz, i.tile_rows, i.tile_cols, i.tiles


def _assert_same_tiled(T, U, tag=""):
    assert _info(T) == _info(U), (tag, _info(T), _info(U))
    for n in ARRAYS:
        x, y = T.array(n), U.array(n)
        if n == "vals":
            _assert_bits(x, y, f"{tag} {n}")
        else:
            assert x.dtype == y.dtype and np.array_equal(x, y), (tag, n)


def _via_coo(ctx, C, transpose=False):
    """The route to_tiled replaces: export C, convert the COO again."""
    r, c, v = C.to_coo()
    i = C.info
    return ctx.convert_coo(i.rows, i.cols, r, c, v, transpose=transpose, dtype=C.dtype)


def _assert_identity(ctx, C, tag=""):
    T, U = C.to_tiled(), _via_coo(ctx, C)
    try:
        _assert_same_tiled(T, U, tag)
    finally:
        T.free()
        U.free()


def _csr(X, f32=False):
    o = host.coo_to_csr(*X)
    if f32:
        o.val = o.val.astype(np.float32).astype(np.float64)
    return o


def _mul(a, b, f32=False):
    return (host.spgemm_f32 if f32 else host.spgemm)(a, b)


def _as64(o):
    """An fp32 oracle result as the next operand of the oracle (its values are exact in fp64)."""
    return host.CSR(o.rows, o.cols, o.ptr, o.idx, o.val.astype(np.float64))


# ---------------------------------------------------------------------------------------------------------------
# 1. identity with the convert route
# ---------------------------------------------------------------------------------------------------------------
def identity_case(ctx, name, f32):
    a, b = CASES[name]
    dt = np.float32 if f32 else np.float64
    A, B = _operands(ctx, a, b, dt)
    try:
        C = ctx.spgemm(A, B)
        _assert_identity(ctx, C, f"{name} {dt.__name__}")
        C.free()
        tr = A.info.tile_rows
        bounds = ctx.partition_panels(A, B, 3)
        for q in range(3):                          # panels: C's full shape, tile rows outside the panel empty
            C = ctx.spgemm(A, B, panel=(bounds[q], bounds[q + 1]))
            _assert_identity(ctx, C, f"{name} {dt.__name__} panel {q}")
            C.free()
        C = ctx.spgemm(A, B, panel=(tr // 3, tr // 3 + 1))
        _assert_identity(ctx, C, f"{name} {dt.__name__} one tile row")
        C.free()
    finally:
        if B is not A:
            B.free()
        A.free()


@pytest.mark.parametrize("f32", [False, True])
@pytest.mark.parametrize("name", list(CASES))
def test_to_tiled_equals_the_convert_route(engine, name, f32):
    identity_case(engine, name, f32)


# ---------------------------------------------------------------------------------------------------------------
# 2. shapes and edge cases
# ---------------------------------------------------------------------------------------------------------------
def test_ragged_shapes(engine):
    rng = np.random.default_rng(3)
    a = _rand_tiled(37, 301, 25, (3, 12), rng)
    b = _rand_tiled(301, 203, 60, (1, 20), rng)
    A, B = engine.convert_coo(*a), engine.convert_coo(*b)
    C = engine.spgemm(A, B)
    T = C.to_tiled()
    assert (T.info.rows, T.info.cols, T.info.tile_rows, T.info.tile_cols) == (37, 203, 3, 13)
    _assert_identity(engine, C, "37 x 203")
    for h in (T, C, A, B):
        h.free()


def test_empty_results(engine):
    rows, cols, I, J, V = synth.random_sparse(40, 50, 200, seed=4)
    A = engine.convert_coo(rows, cols, I, J, V)
    Z = engine.convert_coo(50, 23, np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0))
    C = engine.spgemm(A, Z)
    assert C.info.nnz == 0
    _assert_identity(engine, C, "nnz 0")
    T = C.to_tiled()
    assert _info(T) == (40, 23, 0, 3, 2, 0)
    assert np.array_equal(T.array("tile_row_ptr"), np.zeros(4, np.int32))
    Y = engine.convert_coo(*synth.random_sparse(23, 9, 50, seed=5))
    D = engine.spgemm(T, Y)                          # an empty operand of a product
    assert D.info.nnz == 0
    for h in (D, Y, T, C):
        h.free()
    At = engine.transpose(A)
    for p in ((1, 1), (0, 0), (3, 3)):               # empty panels: the whole matrix is empty
        C = engine.spgemm(A, At, panel=p)
        assert C.info.nnz == 0
        _assert_identity(engine, C, f"panel {p}")
        C.free()
    for h in (At, Z, A):
        h.free()


def test_explicit_zeros_stay(engine):
    MA, MB = Mat(3, 2), Mat(2, 18)
    MA.put(0, 0, 1.0); MA.put(0, 1, 1.0); MA.put(2, 1, 2.0)
    MB.put(0, 0, 1.0); MB.put(1, 0, -1.0); MB.put(1, 17, 0.5)
    a, b = MA.coo(), MB.coo()
    A, B = engine.convert_coo(*a), engine.convert_coo(*b)
    C = engine.spgemm(A, B)
    T = C.to_tiled()
    assert T.info.nnz == 4                           # C(0, 0) = 1 - 1 cancels and stays
    v = T.array("vals")
    assert v[0] == 0 and not np.signbit(v[0])
    _assert_identity(engine, C, "cancellation")
    Tt = engine.transpose(T)
    D = engine.spgemm(T, Tt)
    oC = _mul(_csr(a), _csr(b))
    _assert_result(D, _mul(oC, host.transpose(oC)), "chain through a zero")
    for h in (D, Tt, T, C, A, B):
        h.free()


@pytest.mark.parametrize("fmt", ["f64", "f32"])
@pytest.mark.parametrize("p,dense", [(13, False), (145, True)])
def test_special_values_carried_through(engine, fmt, p, dense):
    f = F64 if fmt == "f64" else F32
    f32 = fmt == "f32"
    dt = np.float32 if f32 else np.float64
    MA, MB = pair_family(p, 3, dense=dense, fmt=f)
    a, b = MA.coo(), MB.coo()
    A, B = engine.convert_coo(*a, dtype=dt), engine.convert_coo(*b, dtype=dt)
    C = engine.spgemm(A, B)
    v = C.array("vals")
    assert np.isnan(v).any() and np.isinf(v).any() and (np.signbit(v) & (v == 0)).any()
    _assert_identity(engine, C, f"witnesses {fmt}")
    T = C.to_tiled()
    _assert_bits(T.array("vals"), v)
    for h in (T, C, A, B):
        h.free()


# ---------------------------------------------------------------------------------------------------------------
# 3. keep-empty results
# ---------------------------------------------------------------------------------------------------------------
def _reachable_empty_tile():
    """C' tile (0, 1) is reached by (A tile (0, 0), B tile (0, 1)) but their product is empty (A column 0, B row 1)."""
    MA, MB = Mat(16, 32), Mat(32, 32)
    MA.put(0, 0, 1.0); MA.put(0, 16, 2.0); MA.put(5, 17, -1.5)
    MB.put(1, 0, 3.0); MB.put(16, 0, 4.0); MB.put(1, 16, 5.0); MB.put(17, 3, 0.25)
    return MA.coo(), MB.coo()


@pytest.mark.parametrize("name", ["constructed", "config2", "config3", "config5", "hyper_x_dense"])
def test_keep_empty_results_drop_their_empty_tiles(engine, name):
    if name == "constructed":
        a, b = _reachable_empty_tile()
    else:
        a, b = CASES[name]
    A, B = _operands(engine, a, b, np.float64)
    try:
        C = engine.spgemm(A, B)
        with Opts(engine, keep_empty_tiles=1):
            K = engine.spgemm(A, B)
            K3 = engine.spgemm(A, B, panel=(0, max(1, A.info.tile_rows // 2)))
        T, U = C.to_tiled(), K.to_tiled()
        _assert_same_tiled(U, T, f"{name} keep-empty")
        _assert_identity(engine, K3, f"{name} keep-empty panel")
        if name == "constructed":
            assert U.info.tiles < K.info.tiles
        assert U.info.tiles == C.info.tiles <= K.info.tiles
        for h in (T, U, C, K, K3):
            h.free()
    finally:
        if B is not A:
            B.free()
        A.free()


# ---------------------------------------------------------------------------------------------------------------
# 4. chains against the host oracle
# ---------------------------------------------------------------------------------------------------------------
def _rect():
    rng = np.random.default_rng(77)
    a = _rand_tiled(37, 301, 30, (4, 16), rng)
    b = _rand_tiled(301, 203, 80, (1, 12), rng)
    d = _rand_tiled(203, 45, 20, (2, 10), rng)
    e = _rand_tiled(50, 37, 8, (3, 9), rng)
    return a, b, d, e


def chain_cases(ctx, owners=(0, 1, 2, 3, 4), paths=(0, 1, 2, 5), f32=False):
    """Every owner under the first step-1 path, every other path under the first owner (both products of a chain)."""
    dt = np.float32 if f32 else np.float64
    # A^3 (config 4: dense tiles, config 2: power-law rows) and (A*A^T)*A (config 3)
    for k in (2, 4, 3):
        _, tb, a = synth.config(k, small=True)
        A = ctx.convert_coo(*a, dtype=dt)
        B = ctx.transpose(A) if tb else A
        oA = _csr(a, f32)
        want = _mul(_as64(_mul(oA, host.transpose(oA) if tb else oA, f32)), oA, f32)
        for owner, path in [(o, paths[0]) for o in owners] + [(owners[0], p) for p in paths[1:]]:
            if f32 and owner in (1, 3):
                continue
            with Opts(ctx, owner=owner, step1_path=path):
                C = ctx.spgemm(A, B)
                T = C.to_tiled()
                C.free()
                D = ctx.spgemm(T, A)
                _assert_result(D, want, f"config {k} owner {owner} path {path}")
                D.free()
                T.free()
        if B is not A:
            B.free()
        A.free()
    # rectangular (A*B)*D, and E*(A*B) with the result as the B operand (its column-major view is built from T)
    a, b, d, e = _rect()
    A, B, D, E = (ctx.convert_coo(*x, dtype=dt) for x in (a, b, d, e))
    oAB = _as64(_mul(_csr(a, f32), _csr(b, f32), f32))
    for owner in owners:
        if f32 and owner in (1, 3):
            continue
        with Opts(ctx, owner=owner):
            C = ctx.spgemm(A, B)
            T = C.to_tiled()
            C.free()
            for X, Y, want, tag in ((T, D, _mul(oAB, _csr(d, f32), f32), "(A*B)*D"),
                                    (E, T, _mul(_csr(e, f32), oAB, f32), "E*(A*B)")):
                R = ctx.spgemm(X, Y)
                _assert_result(R, want, f"{tag} owner {owner}")
                R.free()
            T.free()
    for h in (A, B, D, E):
        h.free()


def test_chains_against_the_oracle(engine):
    chain_cases(engine)


def test_chains_fp32(engine):
    chain_cases(engine, owners=(0, 2, 4), paths=(0,), f32=True)


# ---------------------------------------------------------------------------------------------------------------
# 5. panels
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [2, 4])
def test_panel_chains_concatenate_to_the_full_chain(engine, k):
    _, _, a = synth.config(k, small=True)
    A = engine.convert_coo(*a)
    C = engine.spgemm(A, A)
    T = C.to_tiled()
    full = engine.spgemm(T, A).to_coo()
    b = engine.partition_panels(A, A, 3)
    parts = []
    for q in range(3):
        P = engine.spgemm(A, A, panel=(b[q], b[q + 1]))
        TP = P.to_tiled()
        P.free()
        assert _info(TP)[:2] == _info(T)[:2]
        D = engine.spgemm(TP, A, panel=(b[q], b[q + 1]))
        parts.append(D.to_coo())
        for h in (D, TP):
            h.free()
    got = [np.concatenate([p[j] for p in parts]) for j in range(3)]
    assert np.array_equal(got[0], full[0]) and np.array_equal(got[1], full[1])
    _assert_bits(got[2], full[2])
    oA = _csr(a)
    r, c, v = _mul(_mul(oA, oA), oA).to_coo()
    assert np.array_equal(got[0], r) and np.array_equal(got[1], c)
    _assert_bits(got[2], v)
    for h in (T, C, A):
        h.free()


# ---------------------------------------------------------------------------------------------------------------
# 6. transpose
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["config3", "hyper_x_dense", "dense_x_hyper"])
def test_transpose_of_a_result_handle(engine, name):
    a, b = CASES[name]
    A, B = _operands(engine, a, b, np.float64)
    C = engine.spgemm(A, B)
    T = C.to_tiled()
    Tt = engine.transpose(T)
    U = _via_coo(engine, C, transpose=True)
    _assert_same_tiled(Tt, U, name)
    r, c, _ = C.to_coo()
    V = _vals(r.size, 12)
    Tt.set_values(V)
    U.set_values(V)
    _assert_same_tiled(Tt, U, name + " after set_values")
    i = C.info
    W = engine.convert_coo(i.rows, i.cols, r, c, V, transpose=True)
    _assert_bits(Tt.array("vals"), W.array("vals"))
    for h in (W, U, Tt, T, C):
        h.free()
    if B is not A:
        B.free()
    A.free()


# ---------------------------------------------------------------------------------------------------------------
# 7. lifetime
# ---------------------------------------------------------------------------------------------------------------
def test_handle_outlives_its_result(engine):
    _, _, a = synth.config(4, small=True)
    A = engine.convert_coo(*a)
    C = engine.spgemm(A, A)
    T = C.to_tiled()
    C.free()
    engine.spgemm(A, A).free()                      # C's blocks go back to the cache and are taken again
    D = engine.spgemm(T, A)
    oA = _csr(a)
    _assert_result(D, _mul(_mul(oA, oA), oA), "after the result was freed")
    for h in (D, T, A):
        h.free()


def test_handle_from_a_graph_borrowed_result(engine):
    _, _, a = synth.config(1, small=True)
    A = engine.convert_coo(*a)
    try:
        for _ in range(2):                          # records the size plan, then captures the graph
            engine.spgemm(A, A).free()
        g = engine.graph_replays
        C = engine.spgemm(A, A)
        assert engine.graph_replays == g + 1
        T = C.to_tiled()
        before = {n: T.array(n) for n in ARRAYS}
        C.free()
        V = _vals(a[2].size, 13)
        A.set_values(V)                             # the graph's next run writes other values into its arena
        C2 = engine.spgemm(A, A)
        assert engine.graph_replays == g + 2
        _assert_result(C2, _mul(_csr(_with(a, V)), _csr(_with(a, V))))
        for n, x in before.items():
            y = T.array(n)
            if n == "vals":
                _assert_bits(y, x, n)
            else:
                assert np.array_equal(x, y), n
        oA = _csr(a)
        D = engine.spgemm(T, engine.convert_coo(*a))
        _assert_result(D, _mul(_mul(oA, oA), oA), "graph-borrowed source")
        for h in (D, C2, T):
            h.free()
    finally:
        A.free()


# ---------------------------------------------------------------------------------------------------------------
# 8. numeric chain
# ---------------------------------------------------------------------------------------------------------------
def numeric_chain(ctx, k, steps=3):
    """set_values(A); numeric(A, A, C); T.refresh_from(C); numeric(T, A, D) and numeric(A, T, E), with T's
    column-major view (E: T as B) built before the first refresh."""
    _, _, a = synth.config(k, small=True)
    A = ctx.convert_coo(*a)
    C = ctx.spgemm(A, A)
    T = C.to_tiled()
    D, E = ctx.spgemm(T, A), ctx.spgemm(A, T)
    vptr = pem.load().pem_tiled_device_ptr(T._h, 0)
    for step in range(steps):
        V = _vals(a[2].size, 200 + 10 * k + step)
        A.set_values(V)
        ctx.spgemm_numeric(A, A, C)
        T.refresh_from(C)
        ctx.spgemm_numeric(T, A, D)
        ctx.spgemm_numeric(A, T, E)
        oA = _csr(_with(a, V))
        oC = _mul(oA, oA)
        _assert_result(D, _mul(oC, oA), f"config {k} step {step} T*A")
        _assert_result(E, _mul(oA, oC), f"config {k} step {step} A*T")
        # the full chain of the same values, from a fresh conversion
        F = ctx.convert_coo(*_with(a, V))
        FC = ctx.spgemm(F, F)
        FT = FC.to_tiled()
        _assert_same_tiled(T, FT, f"config {k} step {step} refreshed handle")
        FD = ctx.spgemm(FT, F)
        _assert_bits(D.array("vals"), FD.array("vals"), f"config {k} step {step} full chain")
        for h in (FD, FT, FC, F):
            h.free()
        assert pem.load().pem_tiled_device_ptr(T._h, 0) == vptr
    # the numeric chain alone stalls nowhere (the fresh chains above do)
    s1 = ctx.size_stalls
    for step in range(2):
        A.set_values(_vals(a[2].size, 300 + step))
        ctx.spgemm_numeric(A, A, C)
        T.refresh_from(C)
        ctx.spgemm_numeric(T, A, D)
        ctx.spgemm_numeric(A, T, E)
    assert ctx.size_stalls == s1
    # products that take T replay their graph after a refresh and read the refreshed values
    for _ in range(2):
        ctx.spgemm(T, A).free()
    V = _vals(a[2].size, 400 + k)
    A.set_values(V)
    ctx.spgemm_numeric(A, A, C)
    T.refresh_from(C)
    g, s = ctx.graph_replays, ctx.size_stalls
    G = ctx.spgemm(T, A)
    assert ctx.graph_replays == g + 1 and ctx.size_stalls == s
    oA = _csr(_with(a, V))
    _assert_result(G, _mul(_mul(oA, oA), oA), f"config {k} graph after refresh")
    for h in (G, D, E, T, C, A):
        h.free()


@pytest.mark.parametrize("k", [1, 2, 4])
def test_numeric_chain(engine, k):
    numeric_chain(engine, k)


# ---------------------------------------------------------------------------------------------------------------
# 9. refusals
# ---------------------------------------------------------------------------------------------------------------
def _refused(code, fn, *args):
    with pytest.raises(pem.PemError) as e:
        fn(*args)
    assert e.value.code == code, str(e.value)


def test_refusals_leave_nothing_behind():
    ctx = pem.Context(0)
    try:
        _, _, a = synth.config(1, small=True)
        A, A2 = ctx.convert_coo(*a), ctx.convert_coo(*a)
        S = ctx.step1(A, A)
        ctx.step2(A, A, S)
        _refused(ARG, S.to_tiled)                                       # step 2 only
        C = ctx.spgemm(A, A)
        T = C.to_tiled()
        Tt = ctx.transpose(T)
        O = ctx.spgemm(A, A2)                                           # same shape and values, other product
        P = ctx.spgemm(A, A, panel=(0, 1))                              # same operands, other panel
        _refused(ARG, T.refresh_from, O)
        _refused(ARG, T.refresh_from, P)
        _refused(ARG, A.refresh_from, C)                                # a converted handle
        _refused(ARG, Tt.refresh_from, C)                               # the transpose of a result handle
        _refused(ARG, T.refresh_from, S)                                # an incomplete result of the same product
        C2 = ctx.spgemm(A, A)                                           # any complete result of the product is accepted
        T.refresh_from(C2)
        oA = _csr(a)
        D = ctx.spgemm(T, A)
        _assert_result(D, _mul(_mul(oA, oA), oA), "after the refusals")
        for h in (D, C2, P, O, Tt, T, C, S, A, A2):
            h.free()
        ctx.trim()
        assert ctx.pool_bytes == 0
    finally:
        ctx.close()


# ---------------------------------------------------------------------------------------------------------------
# 10. poisoned memory
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("pattern", [0x00, 0xFF, 0x5A])
def test_under_poisoned_memory(pattern):
    ctx = pem.Context(0)
    try:
        ctx.set_option(pem.OPT_POISON, 0x100 | pattern)
        for name in CASES:
            identity_case(ctx, name, False)
        identity_case(ctx, "config2", True)
        chain_cases(ctx, owners=(0, 3), paths=(0,))
        with Opts(ctx, keep_empty_tiles=1):
            a, b = _reachable_empty_tile()
            A, B = ctx.convert_coo(*a), ctx.convert_coo(*b)
            C = ctx.spgemm(A, B)
            _assert_identity(ctx, C, "keep-empty")
            for h in (C, A, B):
                h.free()
        numeric_chain(ctx, 4, steps=2)
    finally:
        ctx.close()
