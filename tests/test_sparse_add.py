"""Sums of tiled matrices: Context.add (pem_tiled_add) builds S = alpha*A + beta*B on the device as a tiled operand,
Context.add_values (pem_tiled_add_values) recomputes its values in place.

The host oracle ``oracle_add`` below gives the union pattern in (row, col) order with the values of the contract:
fl(fl(alpha*a) + fl(beta*b)) where both operands hold the entry, fl(alpha*a) or fl(beta*b) where one does (numpy's
elementwise float operations round separately; there is no fused multiply-add).  scipy's alpha*A + beta*B is not an
oracle for this: it drops the entries that cancel.  Every structure is compared array for array with what
convert_coo builds from the oracle's COO, every value bit for bit (the sign of zero counts, a NaN matches any NaN)."""
import ctypes
from fractions import Fraction

import numpy as np
import pytest
import scipy.sparse as sp

import pem_spgemm_b200 as pem
from oracle import host
from pem_spgemm_b200 import synth
from test_general_product import F32, F64, Mat, Opts, _assert_bits, _rand_tiled

gpu = pytest.mark.gpu
ARG = -2
ALPHA_BETA = [(1.0, 1.0), (1.0, -1.0), (0.5, -3.0), (0.0, 1.0)]


# ---------------------------------------------------------------------------------------------------------------
# the host oracle
# ---------------------------------------------------------------------------------------------------------------
def oracle_add(a, b, alpha, beta, f32=False):
    """S = alpha*A + beta*B from COO tuples (rows, cols, I, J, V) of the same shape -> (rows, cols, I, J, V) of S,
    sorted by (row, col), on the union of the patterns.  fp32: the values and alpha, beta rounded to float first."""
    rows, cols = a[0], a[1]
    assert (b[0], b[1]) == (rows, cols)
    dt = np.float32 if f32 else np.float64
    al, be = dt(alpha), dt(beta)
    ka = a[2].astype(np.int64) * cols + a[3]
    kb = b[2].astype(np.int64) * cols + b[3]
    keys = np.union1d(ka, kb)
    ia, ib = np.searchsorted(keys, ka), np.searchsorted(keys, kb)
    in_a = np.zeros(keys.size, bool); in_a[ia] = True
    in_b = np.zeros(keys.size, bool); in_b[ib] = True
    with np.errstate(all="ignore"):                 # 0 * Inf and Inf - Inf are NaN on purpose
        pa = np.zeros(keys.size, dt); pa[ia] = np.asarray(a[4]).astype(dt) * al
        pb = np.zeros(keys.size, dt); pb[ib] = np.asarray(b[4]).astype(dt) * be
        v = np.where(in_a, pa, pb)
        both = in_a & in_b
        v[both] = pa[both] + pb[both]
    return rows, cols, (keys // max(cols, 1)).astype(np.int32), (keys % max(cols, 1)).astype(np.int32), v


def _bits(x, dt):
    return np.array([x], dt).view(np.uint32 if dt == np.float32 else np.uint64)[0]


def _one(a_val, b_val, alpha, beta, f32, where="both"):
    """The oracle on one entry held by both operands (or by one)."""
    e = (np.zeros(1, np.int32), np.zeros(1, np.int32))
    none = (np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0))
    a = (1, 1, *e, np.array([a_val])) if where in ("both", "a") else (1, 1, *none)
    b = (1, 1, *e, np.array([b_val])) if where in ("both", "b") else (1, 1, *none)
    return oracle_add(a, b, alpha, beta, f32)[4][0]


# ---------------------------------------------------------------------------------------------------------------
# CPU: the oracle itself
# ---------------------------------------------------------------------------------------------------------------
def _dyadic_positive(rows, cols, nnz, seed):
    rng = np.random.default_rng(seed)
    key = np.unique(rng.integers(0, rows * cols, nnz))
    V = rng.integers(1, 8, key.size) * np.exp2(rng.integers(-4, 5, key.size)).astype(np.float64)
    return rows, cols, (key // cols).astype(np.int32), (key % cols).astype(np.int32), V


@pytest.mark.parametrize("m,n,seed", [(37, 530, 1), (400, 203, 2), (1, 17, 3), (33, 1, 4)])
def test_oracle_add_vs_scipy_exact(m, n, seed):
    """Positive dyadic values and positive alpha, beta: no entry cancels and every sum is exact, so scipy's sum is
    the oracle's, pattern and values."""
    a = _dyadic_positive(m, n, max(1, m * n // 5), seed)
    b = _dyadic_positive(m, n, max(1, m * n // 7), seed + 50)
    for alpha, beta in ((1.0, 1.0), (0.5, 3.0), (2.0, 0.25)):
        rows, cols, I, J, V = oracle_add(a, b, alpha, beta)
        R = (alpha * sp.csr_matrix((a[4], (a[2], a[3])), shape=(m, n))
             + beta * sp.csr_matrix((b[4], (b[2], b[3])), shape=(m, n))).tocoo()
        o = np.lexsort((R.col, R.row))
        assert np.array_equal(I, R.row[o]) and np.array_equal(J, R.col[o])
        _assert_bits(V, R.data[o].astype(np.float64))
        assert np.all(np.diff(I.astype(np.int64) * n + J) > 0)            # (row, col) order, no duplicate


@pytest.mark.parametrize("f32", [False, True])
def test_oracle_add_hand_derived_bits(f32):
    dt = np.float32 if f32 else np.float64
    z = _one(1.5, 1.5, 1.0, -1.0, f32)                                  # cancellation: +0.0, kept
    assert z == 0 and not np.signbit(z)
    z = _one(-0.0, -0.0, 1.0, 1.0, f32)                                 # (-0) + (-0) = -0
    assert z == 0 and np.signbit(z)
    z = _one(-0.0, 0.0, 1.0, 1.0, f32)                                  # (-0) + (+0) = +0
    assert z == 0 and not np.signbit(z)
    z = _one(2.0, 0.0, 0.0, 1.0, f32, where="a")                        # alpha = 0 on a one-sided entry: +0, kept
    assert z == 0 and not np.signbit(z)
    z = _one(-2.0, 0.0, 0.0, 1.0, f32, where="a")                       # 0 * (-2) = -0: an absent B entry is not +0
    assert z == 0 and np.signbit(z)
    assert np.isnan(_one(np.inf, 1.0, 0.0, 1.0, f32))                   # 0 * Inf = NaN
    assert np.isnan(_one(np.inf, np.inf, 1.0, -1.0, f32))               # Inf - Inf = NaN
    assert _one(np.inf, 1.0, 1.0, 1.0, f32, where="a") == np.inf
    w = _one(10.0, 1.0, 0.1, -1.0, f32)                                 # the fused-multiply-add witness
    assert _bits(w, dt) == _bits(0.0, dt)
    # what a fused form would give, the exact alpha*a + beta*b rounded once: 2^-54 in fp64, 2^-26 in fp32
    fused = Fraction(float(dt(0.1))) * 10 - 1
    assert fused == Fraction(2) ** (-26 if f32 else -54)


# ---------------------------------------------------------------------------------------------------------------
# GPU helpers
# ---------------------------------------------------------------------------------------------------------------
ARRAYS = list(pem.T_ARRAYS)


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


def _t(X):
    rows, cols, I, J, V = X
    o = np.lexsort((I, J))
    return cols, rows, J[o].copy(), I[o].copy(), V[o].copy()


def _with(X, V):
    return (*X[:4], V)


def _vals(n, seed, dt=np.float64):
    return np.random.default_rng(seed).uniform(-1, 1, n).astype(dt)


def _empty(rows, cols):
    return rows, cols, np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0)


def _convert(ctx, X, f32):
    return ctx.convert_coo(*X, dtype=np.float32 if f32 else np.float64)


def _assert_sum(ctx, S, a, b, alpha, beta, f32, tag=""):
    """S is, array for array, what convert_coo builds from the oracle's COO of alpha*a + beta*b."""
    U = _convert(ctx, oracle_add(a, b, alpha, beta, f32), f32)
    try:
        _assert_same_tiled(S, U, tag)
    finally:
        U.free()


def _identity_pair(ctx, A, B, a, b, alpha, beta, f32, tag):
    S = ctx.add(A, B, alpha, beta)
    try:
        _assert_sum(ctx, S, a, b, alpha, beta, f32, tag)
    finally:
        S.free()


def _cases():
    """name -> (A COO, B COO or "T" for A's device transpose or "same" for the same handle)"""
    from test_value_updates import CASES
    c = {}
    rng = np.random.default_rng(11)
    for name, (a, _) in CASES.items():
        if a[0] == a[1]:
            c[f"{name}+T"] = (a, "T")
        ntiles = max(1, len(np.unique((a[2] // 16).astype(np.int64) * 100003 + a[3] // 16)))
        c[f"{name}+rand"] = (a, _rand_tiled(a[0], a[1], ntiles, (1, 12), rng))
    _, _, a1 = synth.config(1, small=True)
    c["same_handle"] = (a1, "same")
    # tile-disjoint: A in even tile columns, B in odd ones
    MA, MB = Mat(64, 96), Mat(64, 96)
    for I in range(4):
        for J in range(6):
            M = MA if J % 2 == 0 else MB
            for r in range(0, 16, 3):
                M.tile(I, J, r, (r * 7 + J) % 16, 1.0 + r + 16 * J)
    c["tile_disjoint"] = (MA.coo(), MB.coo())
    # the same tiles, disjoint entries inside them (checkerboard)
    MA, MB = Mat(48, 48), Mat(48, 48)
    for I in range(3):
        for J in range(3):
            if (I + J) % 2 == 0:
                for r in range(16):
                    for cc in range(0, 16, 2):
                        (MA if (r + cc // 2) % 2 else MB).tile(I, J, r, cc + (r % 2), float(r - cc) + 0.25)
    c["same_tiles_disjoint_entries"] = (MA.coo(), MB.coo())
    # A a subset of B
    rows, cols, I, J, V = synth.random_sparse(100, 77, 900, seed=21)
    keep = np.random.default_rng(22).random(I.size) < 0.4
    c["a_subset_of_b"] = ((rows, cols, I[keep], J[keep], V[keep]), (rows, cols, I, J, _vals(I.size, 23)))
    # A - sigma*I
    _, _, a4 = synth.config(4, small=True)
    n = a4[0]
    c["a_shift"] = (a4, (n, n, np.arange(n, dtype=np.int32), np.arange(n, dtype=np.int32), np.ones(n)))
    # empty operands
    c["empty_a"] = (_empty(40, 50), synth.random_sparse(40, 50, 200, seed=4))
    c["empty_b"] = (synth.random_sparse(40, 50, 200, seed=5), _empty(40, 50))
    c["both_empty"] = (_empty(40, 50), _empty(40, 50))
    # tiny and ragged shapes
    for m, k in ((1, 1), (1, 17), (33, 1), (17, 33)):
        c[f"{m}x{k}"] = (synth.random_sparse(m, k, max(1, m * k // 2), seed=m + k),
                         synth.random_sparse(m, k, max(1, m * k // 3), seed=m * k + 7))
    # a B-only tile last in its tile row, and one first in the matrix
    MA, MB = Mat(48, 64), Mat(48, 64)
    for I, J in ((0, 1), (0, 2), (1, 0), (1, 1), (2, 2)):
        MA.tile(I, J, I + 1, J + 2, 1.0 + I + J)
    MB.tile(0, 0, 0, 0, 5.0)                         # first tile of the matrix, B only
    MB.tile(0, 3, 15, 15, 6.0)                       # last of tile row 0, B only
    MB.tile(1, 3, 4, 9, 7.0)                         # last of tile row 1, B only
    MB.tile(2, 3, 0, 1, 8.0)                         # last tile of the matrix, B only
    MB.tile(1, 1, 2, 3, -2.0)                        # shared with A
    c["b_only_at_the_ends"] = (MA.coo(), MB.coo())
    return c


SUM_CASES = _cases()


def _operands(ctx, a, b, f32):
    A = _convert(ctx, a, f32)
    if b == "same":
        return A, A, a
    if b == "T":
        return A, ctx.transpose(A), _t(a)
    return A, _convert(ctx, b, f32), b


def identity_sweep(ctx, f32, alpha_beta=ALPHA_BETA, names=None):
    for name in names or SUM_CASES:
        a, b = SUM_CASES[name]
        A, B, bb = _operands(ctx, a, b, f32)
        try:
            for alpha, beta in alpha_beta:
                _identity_pair(ctx, A, B, a, bb, alpha, beta, f32, f"{name} {alpha},{beta} f32={f32}")
        finally:
            if B is not A:
                B.free()
            A.free()


# ---------------------------------------------------------------------------------------------------------------
# 1. identity with the convert route
# ---------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("alpha,beta", ALPHA_BETA)
@pytest.mark.parametrize("f32", [False, True])
def test_add_equals_the_convert_route(engine, f32, alpha, beta):
    identity_sweep(engine, f32, [(alpha, beta)])


@gpu
def test_add_shapes_and_counts(engine):
    a, b = SUM_CASES["b_only_at_the_ends"]
    A, B = engine.convert_coo(*a), engine.convert_coo(*b)
    S = engine.add(A, B, 2.0, -1.0)
    assert _info(S) == (48, 64, 9, 3, 4, 9)                        # one entry of tile (1, 1) is shared
    assert np.array_equal(S.array("tile_row_ptr"), [0, 4, 7, 9])
    assert np.array_equal(S.array("tile_col_idx"), [0, 1, 2, 3, 0, 1, 3, 2, 3])
    E = engine.convert_coo(*_empty(40, 50))
    Z = engine.add(E, E)
    assert _info(Z) == (40, 50, 0, 3, 4, 0)
    assert np.array_equal(Z.array("tile_row_ptr"), np.zeros(4, np.int32))
    for h in (Z, E, S, A, B):
        h.free()


# ---------------------------------------------------------------------------------------------------------------
# 2. special values
# ---------------------------------------------------------------------------------------------------------------
def _special_pair(f):
    """Every pair of special values in an entry both operands hold, and every special value in entries held by A
    only and by B only."""
    sv = [0.0, -0.0, f.tiny, -f.sub_max, np.inf, -np.inf, np.nan, 1.0, -1.0, f.big]
    MA, MB = Mat(40, 200), Mat(40, 200)
    k = 0
    for x in sv:
        for y in sv:
            MA.put(k // 200, k % 200, x); MB.put(k // 200, k % 200, y)
            k += 1
    for x in sv:
        MA.put(k // 200, k % 200, x); k += 1
        MB.put(k // 200, k % 200, x); k += 1
    return MA.coo(), MB.coo()


@gpu
@pytest.mark.parametrize("fmt", ["f64", "f32"])
def test_special_values(engine, fmt):
    f = F64 if fmt == "f64" else F32
    f32 = fmt == "f32"
    a, b = _special_pair(f)
    A, B = _convert(engine, a, f32), _convert(engine, b, f32)
    for alpha, beta in ALPHA_BETA + [(-0.0, 2.0), (np.inf, 1.0), (f.tiny, 0.5)]:
        _identity_pair(engine, A, B, a, b, alpha, beta, f32, f"special {fmt} {alpha},{beta}")
    # the fused-multiply-add witness: alpha = 0.1, a = 10, beta = -1, b = 1 gives +0.0
    one = np.zeros(1, np.int32)
    WA, WB = _convert(engine, (1, 1, one, one, np.array([10.0])), f32), _convert(engine, (1, 1, one, one, np.array([1.0])), f32)
    W = engine.add(WA, WB, 0.1, -1.0)
    w = W.array("vals")
    assert w[0] == 0 and not np.signbit(w[0]), w
    WA.free(); WB.free()
    # explicit zeros and cancellations stay
    S = engine.add(A, B, 1.0, -1.0)
    assert S.info.nnz == len(set(zip(a[2].tolist(), a[3].tolist())) | set(zip(b[2].tolist(), b[3].tolist())))
    for h in (S, W, A, B):
        h.free()


# ---------------------------------------------------------------------------------------------------------------
# 3. as an operand
# ---------------------------------------------------------------------------------------------------------------
def _csr(X):
    return host.coo_to_csr(*X)


def _assert_result(C, oC, tag=""):
    r, c, v = C.to_coo()
    ro, co, vo = oC.to_coo()
    assert np.array_equal(r, ro) and np.array_equal(c, co), tag
    _assert_bits(v, vo.astype(v.dtype), tag)


def operand_cases(ctx, owners=(0, 1, 2, 3, 4), paths=(0, 1, 2, 5)):
    """S*X and X*S against the host oracle, every owner under the first step-1 path, every other path under the first
    owner; S = A - 0.5*A^T (config 2: power-law tile rows; config 4: dense tiles) and X = A."""
    for k in (2, 4):
        _, _, a = synth.config(k, small=True)
        A = ctx.convert_coo(*a)
        At = ctx.transpose(A)
        s = oracle_add(a, _t(a), 1.0, -0.5)
        oS, oA = _csr(s), _csr(a)
        for owner, path in [(o, paths[0]) for o in owners] + [(owners[0], p) for p in paths[1:]]:
            with Opts(ctx, owner=owner, step1_path=path):
                S = ctx.add(A, At, 1.0, -0.5)
                for X, Y, want, tag in ((S, A, host.spgemm(oS, oA), "S*A"), (A, S, host.spgemm(oA, oS), "A*S")):
                    R = ctx.spgemm(X, Y)
                    _assert_result(R, want, f"config {k} {tag} owner {owner} path {path}")
                    R.free()
                S.free()
        At.free()
        A.free()


@gpu
def test_sum_as_an_operand(engine):
    operand_cases(engine)


@gpu
def test_sum_of_a_result_handle_and_of_sums(engine):
    _, _, a = synth.config(1, small=True)
    A = engine.convert_coo(*a)
    C = engine.spgemm(A, A)
    T = C.to_tiled()
    r, c, v = C.to_coo()
    t = (a[0], a[1], r, c, v)
    S = engine.add(T, A, 1.0, 2.0)                                     # T + 2A, T from to_tiled
    _assert_sum(engine, S, t, a, 1.0, 2.0, False, "T + 2A")
    S2 = engine.add(S, A, 0.5, -3.0)                                   # a sum of sums
    _assert_sum(engine, S2, oracle_add(t, a, 1.0, 2.0), a, 0.5, -3.0, False, "(T + 2A)/2 - 3A")
    S3 = engine.add(S2, S2, 1.0, 1.0)
    _assert_sum(engine, S3, oracle_add(oracle_add(t, a, 1.0, 2.0), a, 0.5, -3.0),
                oracle_add(oracle_add(t, a, 1.0, 2.0), a, 0.5, -3.0), 1.0, 1.0, False, "S2 + S2")
    for h in (S3, S2, S, T, C, A):
        h.free()


@gpu
def test_operands_freed_before_the_sum_is_used(engine):
    _, _, a = synth.config(4, small=True)
    b = _rand_tiled(a[0], a[1], 40, (1, 12), np.random.default_rng(5))
    A, B = engine.convert_coo(*a), engine.convert_coo(*b)
    S = engine.add(A, B, 1.0, -2.0)
    A.free(); B.free()
    engine.spgemm(engine.convert_coo(*a), engine.convert_coo(*a)).free()   # the freed blocks are taken again
    s = oracle_add(a, b, 1.0, -2.0)
    _assert_sum(engine, S, a, b, 1.0, -2.0, False, "after free")
    R = engine.spgemm(S, S)
    _assert_result(R, host.spgemm(_csr(s), _csr(s)), "S*S after free")
    R.free()
    S.free()


@gpu
def test_add_waits_for_pending_uploads(engine):
    import torch
    rows, cols, I, J, _ = a = synth.cage_like(80, 80, 80)
    V0, W0 = _vals(I.size, 80), _vals(I.size, 81)
    h = [torch.from_numpy(np.ascontiguousarray(x)).pin_memory() for x in (I, J, V0, W0)]
    torch.cuda.synchronize()
    engine.set_option(pem.OPT_ASYNC_VALUES, 1)
    try:
        A = engine.convert_coo(rows, cols, h[0].data_ptr(), h[1].data_ptr(), h[2].data_ptr(), nnz=I.size)
        B = engine.convert_coo(rows, cols, h[0].data_ptr(), h[1].data_ptr(), h[3].data_ptr(), nnz=I.size,
                               transpose=True)
        S = engine.add(A, B, 1.0, -1.0)                                # both uploads may still be in flight
    finally:
        engine.set_option(pem.OPT_ASYNC_VALUES, 0)
    _assert_sum(engine, S, _with(a, V0), _t(_with(a, W0)), 1.0, -1.0, False, "pending uploads")
    for x in (S, A, B):
        x.free()


# ---------------------------------------------------------------------------------------------------------------
# 4. add_values
# ---------------------------------------------------------------------------------------------------------------
def _dev(V):
    import torch
    d = torch.from_numpy(np.ascontiguousarray(V)).cuda()
    torch.cuda.synchronize()
    return d


def refresh_sweep(ctx, f32, names=("config2+T", "config4+rand", "hyper_x_dense+rand", "same_handle", "a_shift",
                                   "b_only_at_the_ends", "empty_a", "both_empty")):
    """S = add(A, B); then new values of A (host) and B (device) and new or unchanged alpha, beta by add_values:
    S equals a fresh add array for array, its values pointer stays, and nothing is allocated or waited for."""
    dt = np.float32 if f32 else np.float64
    for name in names:
        a, b = SUM_CASES[name]
        A, B, bb = _operands(ctx, a, b, f32)
        try:
            S = ctx.add(A, B, 1.0, -1.0)
            vptr = pem.load().pem_tiled_device_ptr(S._h, 0)
            for step, (alpha, beta) in enumerate([(1.0, -1.0), (0.5, 3.0), (0.1, -0.7), (-2.0, 0.0)]):
                Va = _vals(a[2].size, 500 + step, dt)
                Wb = _vals(bb[2].size, 600 + step, dt)
                A.set_values(Va)                    # from host memory
                if b == "T":                        # one V refreshes A and A^T; from device memory
                    B.set_values(_dev(Va).data_ptr() if Va.size else Va)
                elif B is not A:
                    B.set_values(_dev(Wb).data_ptr() if Wb.size else Wb)
                a_now = _with(a, Va)
                b_now = a_now if b == "same" else _t(a_now) if b == "T" else _with(bb, Wb)
                m, s = ctx.pool_mallocs, ctx.size_stalls
                ctx.add_values(S, A, B, alpha, beta)
                assert ctx.pool_mallocs == m and ctx.size_stalls == s, name
                assert pem.load().pem_tiled_device_ptr(S._h, 0) == vptr
                _assert_sum(ctx, S, a_now, b_now, alpha, beta, f32, f"{name} refresh {step}")
                F = ctx.add(A, B, alpha, beta)
                _assert_same_tiled(S, F, f"{name} fresh {step}")
                F.free()
            S.free()
        finally:
            if B is not A:
                B.free()
            A.free()


@gpu
@pytest.mark.parametrize("f32", [False, True])
def test_add_values_equals_a_fresh_add(engine, f32):
    refresh_sweep(engine, f32)


def graph_refresh(ctx, k=2):
    """X*S with graphs on: capture, refresh S by add_values, replay.  S as B is read through its column-major view,
    which add_values writes."""
    _, _, a = synth.config(k, small=True)
    A = ctx.convert_coo(*a)
    At = ctx.transpose(A)
    S = ctx.add(A, At, 1.0, 1.0)
    X = ctx.convert_coo(*a)
    for _ in range(2):                              # records the size plan, then captures the graph
        ctx.spgemm(X, S).free()
    for step in range(2):
        V = _vals(a[2].size, 700 + step)
        A.set_values(V)
        At.set_values(V)
        ctx.add_values(S, A, At, 0.25, -1.5 - step)
        g, s = ctx.graph_replays, ctx.size_stalls
        R = ctx.spgemm(X, S)
        assert ctx.graph_replays == g + 1 and ctx.size_stalls == s
        s_now = oracle_add(_with(a, V), _t(_with(a, V)), 0.25, -1.5 - step)
        _assert_result(R, host.spgemm(_csr(a), _csr(s_now)), f"graph replay {step}")
        R.free()
    for h in (X, S, At, A):
        h.free()


@gpu
def test_add_values_under_a_product_graph(engine):
    graph_refresh(engine)


# ---------------------------------------------------------------------------------------------------------------
# 5. refusals
# ---------------------------------------------------------------------------------------------------------------
def _refused(code, fn, *args):
    with pytest.raises(pem.PemError) as e:
        fn(*args)
    assert e.value.code == code, str(e.value)


@gpu
def test_refusals_leave_nothing_behind():
    ctx = pem.Context(0)
    try:
        _, _, a = synth.config(1, small=True)
        A, A2 = ctx.convert_coo(*a), ctx.convert_coo(*a)
        At = ctx.transpose(A)
        R = ctx.convert_coo(*synth.random_sparse(a[0], a[1] + 1, 100, seed=3))
        F = ctx.convert_coo(*a, dtype=np.float32)
        _refused(ARG, ctx.add, A, R)                                    # shapes
        _refused(ARG, ctx.add, A, F)                                    # dtypes
        L = pem.load()
        h = ctypes.c_void_p()
        assert L.pem_tiled_add(ctx._h, 1.0, None, 1.0, A._h, ctypes.byref(h)) == ARG
        assert L.pem_tiled_add(ctx._h, 1.0, A._h, 1.0, None, ctypes.byref(h)) == ARG
        assert L.pem_tiled_add(ctx._h, 1.0, A._h, 1.0, A._h, None) == ARG
        assert L.pem_tiled_add_values(ctx._h, None, 1.0, A._h, 1.0, At._h) == ARG
        S = ctx.add(A, At, 1.0, -1.0)
        St = ctx.transpose(S)
        C = ctx.spgemm(A, A)
        T = C.to_tiled()
        _refused(ARG, ctx.add_values, S, At, A)                        # swapped
        _refused(ARG, ctx.add_values, S, A2, At)                       # another handle
        _refused(ARG, ctx.add_values, A, A, At)                        # a converted handle
        _refused(ARG, ctx.add_values, T, A, A)                         # a to_tiled handle
        _refused(ARG, ctx.add_values, St, A, At)                       # the transpose of a sum
        _refused(ARG, S.refresh_from, C)                               # a sum is not a result handle
        ctx.add_values(S, A, At, 2.0, 1.0)
        _assert_sum(ctx, S, a, _t(a), 2.0, 1.0, False, "after the refusals")
        for x in (T, C, St, S, F, R, At, A, A2):
            x.free()
        ctx.trim()
        assert ctx.pool_bytes == 0
    finally:
        ctx.close()


# ---------------------------------------------------------------------------------------------------------------
# 6. poisoned memory
# ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(params=[0x00, 0xFF, 0x5A], ids=lambda p: f"poison{p:02x}")
def poisoned(request):
    ctx = pem.Context(0)
    ctx.set_option(pem.OPT_POISON, 0x100 | request.param)
    yield ctx
    ctx.close()


def _snapshot(ctx, f32):
    """Every array of every sum of the identity sweep (one alpha, beta) and of the refresh sweep's final state."""
    out = {}
    for name in SUM_CASES:
        a, b = SUM_CASES[name]
        A, B, _ = _operands(ctx, a, b, f32)
        S = ctx.add(A, B, 0.5, -3.0)
        out[name] = {n: S.array(n) for n in ARRAYS}
        S.free()
        if B is not A:
            B.free()
        A.free()
    return out


_POISON_SEEN = {}


@gpu
def test_under_poisoned_memory(poisoned):
    identity_sweep(poisoned, False, [(0.5, -3.0)])
    identity_sweep(poisoned, True, [(1.0, -1.0)], names=["config2+T", "b_only_at_the_ends", "1x17"])
    refresh_sweep(poisoned, False)
    graph_refresh(poisoned)
    snap = _snapshot(poisoned, False)
    for prev in _POISON_SEEN.values():              # every array identical across the patterns
        for name, arrs in snap.items():
            for n, x in arrs.items():
                assert np.array_equal(x.view(np.uint8), prev[name][n].view(np.uint8)), (name, n)
    _POISON_SEEN[len(_POISON_SEEN)] = snap
