"""Numeric-only re-multiplication: pem_tiled_set_values refreshes an operand's values in place, pem_spgemm_numeric
recomputes a result's values on its existing structure.

Every comparison is bit for bit against the host oracle run on the NEW values (the sign of zero counts, a NaN matches
any NaN), and every case also checks that a fresh conversion plus product of the new values gives the same arrays.
Values are seeded and differ from one refresh to the next, so a refresh that lands in the wrong slot, misses the
column-major view B's values are read from in step 3, or loses a race with a pending upload shows up as a value
difference."""
import numpy as np
import pytest

import pem_spgemm_b200 as pem
from oracle import host
from pem_spgemm_b200 import synth
from test_general_product import DENSITY, F32, F64, SHAPES, Opts, _assert_bits, _rand_tiled, pair_family

pytestmark = pytest.mark.gpu

R_VALS, T_VALS = 9, 0
ARG = -2


# ---------------------------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------------------------
def _vals(n, seed, dt=np.float64):
    return np.random.default_rng(seed).uniform(-1, 1, n).astype(dt)


def _t(X):
    rows, cols, I, J, V = X
    return cols, rows, J.copy(), I.copy(), V.copy()


def _oracle(a, b, f32=False):
    """C = A*B on the host, from COO tuples."""
    oA, oB = host.coo_to_csr(*a), host.coo_to_csr(*b)
    return (host.spgemm_f32 if f32 else host.spgemm)(oA, oB)


def _with(X, V):
    rows, cols, I, J, _ = X
    return rows, cols, I, J, V


def _assert_result(C, oC, tag=""):
    r, c, v = C.to_coo()
    ro, co, vo = oC.to_coo()
    assert np.array_equal(r, ro) and np.array_equal(c, co), tag
    _assert_bits(v, vo.astype(v.dtype), tag)


def _structure(C):
    return {n: C.array(n) for n in ("row_ptr", "tile_row", "tile_col", "pair_ptr", "pairs_a", "pairs_b", "masks",
                                    "tile_nnz_ptr")}


def _vals_ptr(C):
    return pem.load().pem_result_device_ptr(C._h, R_VALS)


def _tiled_vals_ptr(T):
    return pem.load().pem_tiled_device_ptr(T._h, T_VALS)


def _fresh_equal(ctx, a, b_t, f32, C, tag):
    """A new conversion of the new values and a new product give the arrays the refreshed result holds."""
    dt = np.float32 if f32 else np.float64
    A = ctx.convert_coo(*a, dtype=dt)
    B = ctx.convert_coo(*a, transpose=True, dtype=dt) if b_t == "T" else ctx.convert_coo(*b_t, dtype=dt) if b_t else A
    F = ctx.spgemm(A, B)
    for n in ("tile_col", "masks", "tile_nnz_ptr", "vals"):
        x, y = F.array(n), C.array(n)
        if n == "vals":
            _assert_bits(y, x, f"{tag} fresh {n}")
        else:
            assert np.array_equal(x, y), f"{tag} fresh {n}"
    F.free()
    if B is not A:
        B.free()
    A.free()


def _cases():
    """name -> (A COO, B: None for A*A, "T" for A*A^T, or an independent COO)"""
    c = {}
    for k in range(1, 6):
        _, tb, A = synth.config(k, small=True)
        c[f"config{k}"] = (A, "T" if tb else None)
    for shape, da, db in (("wide", "hyper", "hyper"), ("wide", "hyper", "dense"), ("tall", "dense", "hyper"),
                          ("tall", "dense", "dense")):
        m, k, n, ta, tb = SHAPES[shape]
        rng = np.random.default_rng(sum(map(ord, shape + da + db)))
        c[f"{da}_x_{db}"] = (_rand_tiled(m, k, ta, DENSITY[da], rng), _rand_tiled(k, n, tb, DENSITY[db], rng))
    return c


CASES = _cases()


def _operands(ctx, a, b, dt):
    A = ctx.convert_coo(*a, dtype=dt)
    if b is None:
        return A, A
    if b == "T":
        return A, ctx.transpose(A)
    return A, ctx.convert_coo(*b, dtype=dt)


def _variants(name, f32):
    """(owner, step2 kernel) pairs a case runs: every owner with one step-2 form (list 1 or row-mask 3, alternating
    with the case), plus the automatic choice; fp32 takes the kernels it may run (owners 0, 2, 4)."""
    if f32:
        return [(0, 0), (2, 0), (4, 3)]
    h = sum(map(ord, name)) % 2
    return [(0, 0)] + [(o, 1 if (o + h) % 2 else 3) for o in range(5)]


def run_case(ctx, name, f32, variants=None):
    a, b = CASES[name]
    dt = np.float32 if f32 else np.float64
    V0, V1 = _vals(a[2].size, 1, dt), _vals(a[2].size, 2, dt)
    W0 = W1 = None
    if b not in (None, "T"):
        W0, W1 = _vals(b[2].size, 3, dt), _vals(b[2].size, 4, dt)

    def b_with(Va, Wa):
        return _t(_with(a, Va)) if b == "T" else _with(b, Wa) if W0 is not None else None

    o0 = _oracle(_with(a, V0), b_with(V0, W0) or _with(a, V0), f32)
    o1 = _oracle(_with(a, V1), b_with(V1, W1) or _with(a, V1), f32)
    A, B = _operands(ctx, _with(a, V0), None if b is None else "T" if b == "T" else _with(b, W0), dt)
    kernels = set()
    try:
        for owner, step2 in variants or _variants(name, f32):
            tag = f"{name} {'f32' if f32 else 'f64'} owner {owner} step2 {step2}"
            with Opts(ctx, owner=owner, step2_kernel=step2):
                C = ctx.spgemm(A, B)
                s3 = ctx.last_step3_kernel
                kernels.add(s3)
                _assert_result(C, o0, tag + " before")
                before, ptr = _structure(C), _vals_ptr(C)
                A.set_values(V1)
                if B is not A:
                    B.set_values(V1 if W1 is None else W1)
                ctx.spgemm_numeric(A, B, C)
                assert ctx.last_step3_kernel == s3, tag
                _assert_result(C, o1, tag + " after")
                after = _structure(C)
                for n, x in before.items():
                    assert np.array_equal(x, after[n]), (tag, n)
                assert _vals_ptr(C) == ptr, tag
                if owner == 0:
                    _fresh_equal(ctx, _with(a, V1), b if b in (None, "T") else _with(b, W1), f32, C, tag)
                C.free()
                A.set_values(V0)                        # back to the values the next variant's product starts from
                if B is not A:
                    B.set_values(V0 if W0 is None else W0)
    finally:
        if B is not A:
            B.free()
        A.free()
    return kernels


# ---------------------------------------------------------------------------------------------------------------
# 1. every config and kernel
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(CASES))
def test_refresh_then_numeric_every_kernel(engine, name):
    kernels = run_case(engine, name, False)
    assert {1, 3} <= kernels and kernels & {2, 4}


@pytest.mark.parametrize("name", ["config1", "config2", "config3", "hyper_x_dense", "dense_x_dense"])
def test_refresh_then_numeric_fp32(engine, name):
    run_case(engine, name, True)


def test_numeric_reruns_the_recorded_kernel(engine):
    """A result with hit words (config 2, automatic owner: entry-owner kernel) refreshed after PEM_OPT_OWNER changed
    to the window kernel still runs the entry-owner kernel."""
    a, _ = CASES["config2"]
    A = engine.convert_coo(*a)
    try:
        C = engine.spgemm(A, A)
        assert engine.last_step3_kernel == 2
        V1 = _vals(a[2].size, 7)
        A.set_values(V1)
        with Opts(engine, owner=4):
            engine.spgemm_numeric(A, A, C)
            assert engine.last_step3_kernel == 2
        _assert_result(C, _oracle(_with(a, V1), _with(a, V1)))
        C.free()
    finally:
        A.free()


# ---------------------------------------------------------------------------------------------------------------
# 2. input orders
# ---------------------------------------------------------------------------------------------------------------
def _assert_map(T, V):
    pos = T.array("val_pos")
    assert np.array_equal(np.sort(pos), np.arange(pos.size, dtype=np.uint32))
    _assert_bits(T.array("vals"), V[pos])


def input_orders(ctx):
    import torch
    rows, cols, I, J, _ = synth.random_sparse(300, 200, 3000, seed=11)
    p = np.random.default_rng(5).permutation(I.size)
    X = (rows, cols, I[p].copy(), J[p].copy(), _vals(I.size, 20))            # shuffled host COO
    V1 = _vals(I.size, 21)
    want = _oracle(_with(X, V1), _t(_with(X, V1)))

    # host COO, its device transpose and a transposed conversion: one V1 for A and A^T
    A = ctx.convert_coo(*X)
    At = ctx.transpose(A)
    At2 = ctx.convert_coo(*X, transpose=True)
    assert np.array_equal(At.array("val_pos"), At2.array("val_pos"))
    C, C2 = ctx.spgemm(A, At), ctx.spgemm(A, At2)
    for T in (A, At, At2):
        T.set_values(V1)
        _assert_map(T, V1)
    ctx.spgemm_numeric(A, At, C)
    ctx.spgemm_numeric(A, At2, C2)
    _assert_result(C, want, "A*A^T device transpose")
    _assert_result(C2, want, "A*A^T transposed conversion")
    _fresh_equal(ctx, _with(X, V1), "T", False, C, "A*A^T")
    for h in (C, C2, A, At, At2):
        h.free()

    # device COO, refreshed from a device array
    d = [torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in X[2:]]
    dV1 = torch.from_numpy(V1).cuda()
    torch.cuda.synchronize()
    A = ctx.convert_coo(rows, cols, *(t.data_ptr() for t in d), nnz=I.size)
    B = ctx.convert_coo(*_t(X))
    C = ctx.spgemm(A, B)
    A.set_values(dV1.data_ptr())
    B.set_values(V1)
    ctx.spgemm_numeric(A, B, C)
    _assert_map(A, V1)
    _assert_result(C, want, "device COO")
    for h in (C, A, B):
        h.free()

    # host CSR with unsorted columns inside its rows
    o = host.coo_to_csr(*X)
    col = o.idx.copy()
    q = np.arange(col.size)
    rng = np.random.default_rng(9)
    for r in range(rows):
        s, e = o.ptr[r], o.ptr[r + 1]
        q[s:e] = s + rng.permutation(e - s)
    col = col[q]
    W0, W1 = _vals(col.size, 30), _vals(col.size, 31)
    A = ctx.convert_csr(rows, cols, o.ptr.astype(np.int32), col, W0)
    At = ctx.transpose(A)
    C = ctx.spgemm(A, At)
    A.set_values(W1)
    At.set_values(W1)
    ctx.spgemm_numeric(A, At, C)
    _assert_map(A, W1)
    Icsr = np.repeat(np.arange(rows, dtype=np.int32), np.diff(o.ptr))
    Y = (rows, cols, Icsr, col, W1)
    _assert_result(C, _oracle(Y, _t(Y)), "CSR unsorted columns")
    for h in (C, A, At):
        h.free()


def test_refresh_follows_every_input_order(engine):
    input_orders(engine)


# ---------------------------------------------------------------------------------------------------------------
# 3. A^2 with one handle
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [2, 4])
def test_square_with_one_handle(engine, k):
    """One refresh serves A in both roles, including the column-major view B's values are read from."""
    _, _, a = synth.config(k, small=True)
    A = engine.convert_coo(*a)
    try:
        C = engine.spgemm(A, A)
        for seed in (41, 42):
            V = _vals(a[2].size, seed)
            A.set_values(V)
            engine.spgemm_numeric(A, A, C)
            _assert_result(C, _oracle(_with(a, V), _with(a, V)), f"seed {seed}")
        _fresh_equal(engine, _with(a, V), None, False, C, "A^2")
        C.free()
    finally:
        A.free()


# ---------------------------------------------------------------------------------------------------------------
# 4. full products after a refresh: same plan, same graph, new values
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [1, 4])
def test_full_products_after_refresh_replay_their_graph(engine, k):
    _, _, a = synth.config(k, small=True)
    A = engine.convert_coo(*a)
    try:
        for _ in range(2):                          # records the size plan, then captures the graph
            engine.spgemm(A, A).free()
        ptr = _tiled_vals_ptr(A)
        A.set_values(_vals(a[2].size, 50))
        assert _tiled_vals_ptr(A) == ptr
        for step in range(3):
            V = _vals(a[2].size, 60 + step)
            A.set_values(V)
            s, g = engine.size_stalls, engine.graph_replays
            C = engine.spgemm(A, A)
            assert engine.size_stalls == s and engine.graph_replays == g + 1, step
            _assert_result(C, _oracle(_with(a, V), _with(a, V)), f"step {step}")
            C.free()
        assert _tiled_vals_ptr(A) == ptr
    finally:
        A.free()


# ---------------------------------------------------------------------------------------------------------------
# 5. panels
# ---------------------------------------------------------------------------------------------------------------
def test_panels_refresh_their_own_rows(engine):
    _, _, a = synth.config(2, small=True)
    A = engine.convert_coo(*a)
    try:
        b = engine.partition_panels(A, A, 3)
        Cs = [engine.spgemm(A, A, panel=(b[q], b[q + 1])) for q in range(3)]
        V = _vals(a[2].size, 70)
        A.set_values(V)
        parts = []
        for C in Cs:
            engine.spgemm_numeric(A, A, C)
            parts.append(C.to_coo())
            C.free()
        got = [np.concatenate([p[j] for p in parts]) for j in range(3)]
        r, c, v = _oracle(_with(a, V), _with(a, V)).to_coo()
        assert np.array_equal(got[0], r) and np.array_equal(got[1], c)
        _assert_bits(got[2], v)
    finally:
        A.free()


# ---------------------------------------------------------------------------------------------------------------
# 6. a refresh while the conversion's value upload is still pending
# ---------------------------------------------------------------------------------------------------------------
def async_refresh(ctx):
    """A refresh issued right after an asynchronous conversion (78 MB of values from pinned memory) must win over the
    conversion's gather of the old values, however far that gather has got."""
    import torch
    rows, cols, I, J, _ = a = synth.cage_like(80, 80, 80)
    V0, V1 = _vals(I.size, 80), _vals(I.size, 81)
    h = [torch.from_numpy(np.ascontiguousarray(x)).pin_memory() for x in (I, J, V0)]
    dV1 = torch.from_numpy(V1).cuda()               # a device V: the refresh kernel is queued at once
    torch.cuda.synchronize()
    ctx.set_option(pem.OPT_ASYNC_VALUES, 1)
    try:
        A = ctx.convert_coo(rows, cols, *(t.data_ptr() for t in h), nnz=I.size)
        A.set_values(dV1.data_ptr())                # before values_ready
    finally:
        ctx.set_option(pem.OPT_ASYNC_VALUES, 0)
    A.values_ready()
    _assert_map(A, V1)
    C = ctx.spgemm(A, A)
    _fresh_equal(ctx, _with(a, V1), None, False, C, "after a pending upload")
    C.free()
    A.free()


def test_refresh_waits_for_a_pending_upload(engine):
    async_refresh(engine)


# ---------------------------------------------------------------------------------------------------------------
# 7. special values
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fmt", ["f64", "f32"])
@pytest.mark.parametrize("p,dense", [(13, False), (145, True)])
def test_refresh_to_special_values(engine, fmt, p, dense):
    """Random values first, then the order witnesses of test_general_product (+-0, subnormals, Inf, NaN) by refresh;
    then A refreshed to zeros: every entry stays in C and holds +0.0."""
    f = F64 if fmt == "f64" else F32
    MA, MB = pair_family(p, 3, dense=dense, fmt=f)
    a, b = MA.coo(), MB.coo()
    f32 = fmt == "f32"
    dt = np.float32 if f32 else np.float64
    A = engine.convert_coo(*_with(a, _vals(a[2].size, 90, dt)), dtype=dt)
    B = engine.convert_coo(*_with(b, _vals(b[2].size, 91, dt)), dtype=dt)
    try:
        C = engine.spgemm(A, B)
        A.set_values(a[4].astype(dt))
        B.set_values(b[4].astype(dt))
        engine.spgemm_numeric(A, B, C)
        _assert_result(C, _oracle(a, b, f32), "witnesses")
        _fresh_equal(engine, a, b, f32, C, "witnesses")
        B.set_values(_vals(b[2].size, 92, dt))
        A.set_values(np.zeros(a[2].size, dt))
        nnz = C.info.nnz
        engine.spgemm_numeric(A, B, C)
        v = C.array("vals")
        assert C.info.nnz == nnz and v.size == nnz
        assert np.array_equal(v.view(np.uint32 if f32 else np.uint64), np.zeros(nnz, v.view(np.uint32 if f32 else np.uint64).dtype))
        C.free()
    finally:
        A.free(); B.free()


# ---------------------------------------------------------------------------------------------------------------
# 8. refusals
# ---------------------------------------------------------------------------------------------------------------
def _refused(code, fn, *args):
    with pytest.raises(pem.PemError) as e:
        fn(*args)
    assert e.value.code == code, str(e.value)


def test_refusals_leave_nothing_behind():
    ctx = pem.Context(0)
    try:
        L = pem.load()
        _, _, a = synth.config(1, small=True)
        A1, A2 = ctx.convert_coo(*a), ctx.convert_coo(*a)
        C = ctx.spgemm(A1, A1)
        _refused(ARG, ctx.spgemm_numeric, A2, A2, C)                   # same shape, other handles
        _refused(ARG, ctx.spgemm_numeric, A1, A2, C)
        S = ctx.step1(A1, A1)
        ctx.step2(A1, A1, S)
        _refused(ARG, ctx.spgemm_numeric, A1, A1, S)                   # stage 2
        F = ctx.convert_coo(*a, dtype=np.float32)
        V = np.ones(a[2].size)
        _refused(ARG, lambda: ctx._check(L.pem_tiled_set_values(ctx._h, F._h, pem._ptr(V))))        # fp64 into fp32
        _refused(ARG, lambda: ctx._check(L.pem_tiled_set_values_f32(ctx._h, A1._h, pem._ptr(V.astype(np.float32)))))
        _refused(ARG, A1.set_values, None)                             # null V
        Z = ctx.convert_coo(16, 16, np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0))
        Z.set_values(None)                                             # nnz == 0: a no-op
        ctx.spgemm_numeric(A1, A1, C)                                  # the refusals changed nothing
        _assert_result(C, _oracle(a, a))
        for h in (C, S, A1, A2, F, Z):
            h.free()
        ctx.trim()
        assert ctx.pool_bytes == 0
    finally:
        ctx.close()


# ---------------------------------------------------------------------------------------------------------------
# 9. poisoned memory
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("pattern", [0xFF, 0x5A])
def test_refresh_under_poisoned_memory(pattern):
    ctx = pem.Context(0)
    try:
        ctx.set_option(pem.OPT_POISON, 0x100 | pattern)
        for name in ("config4", "config2"):
            run_case(ctx, name, False, variants=[(0, 0), (2, 1), (3, 3)])
        input_orders(ctx)
        async_refresh(ctx)
    finally:
        ctx.close()


# ---------------------------------------------------------------------------------------------------------------
# 10. steady state
# ---------------------------------------------------------------------------------------------------------------
def test_refresh_loop_allocates_nothing_new(engine):
    import torch
    _, _, a = synth.config(4, small=True)
    A = engine.convert_coo(*a)
    try:
        C = engine.spgemm(A, A)
        dV = torch.from_numpy(_vals(a[2].size, 100)).cuda()
        torch.cuda.synchronize()
        m = None
        for step in range(6):
            V = _vals(a[2].size, 101 + step)
            if step % 2:
                dV.copy_(torch.from_numpy(V))
                torch.cuda.synchronize()
                A.set_values(dV.data_ptr())
            else:
                A.set_values(V)
            engine.spgemm_numeric(A, A, C)
            if step == 1:
                m = engine.pool_mallocs
            elif step > 1:
                assert engine.pool_mallocs == m, step
        _assert_result(C, _oracle(_with(a, V), _with(a, V)))
        C.free()
    finally:
        A.free()
