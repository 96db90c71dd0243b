"""A refused call returns every device block it took, and a stage retried after a refusal neither leaks nor
overwrites a live buffer.  Each case runs in a context of its own; after the refusal the same context multiplies one
product bit for bit against the host oracle, and once every handle is freed and the cache trimmed, the context's pool
holds no memory at all."""
import numpy as np
import pytest

import pem_spgemm_b200 as pem
from oracle import host
from pem_spgemm_b200 import synth
from test_general_product import _assert_bits, hash_row_case

pytestmark = pytest.mark.gpu

LAP = synth.laplacian2d(24)          # dense tiles: step 2 runs in dense-tile mode under the default options


@pytest.fixture
def ctx():
    c = pem.Context(0)
    yield c
    c.close()


def _assert_same(C, oC):
    r, c, v = C.to_coo()
    ro, co, vo = oC.to_coo()
    assert np.array_equal(r, ro) and np.array_equal(c, co)
    _assert_bits(v, vo)


def _clean_product(ctx):
    """One product after the refusal, in the same context: A*A bit for bit against the host oracle."""
    rows, cols, I, J, V = LAP
    A = ctx.convert_coo(rows, cols, I, J, V)
    C = ctx.spgemm(A, A)
    _assert_same(C, host.spgemm_from_coo(rows, cols, I, J, V, False)[2])
    C.free()
    A.free()


def _assert_nothing_held(ctx):
    ctx.trim()
    assert ctx.pool_bytes == 0


def _refused(code, fn, *args):
    with pytest.raises(pem.PemError) as e:
        fn(*args)
    assert e.value.code == code, str(e.value)


def test_clean_product_leaves_nothing(ctx):
    _clean_product(ctx)
    _assert_nothing_held(ctx)


def test_step2_fp32_refused_under_owner_3_and_1_then_retried(ctx):
    rows, cols, I, J, V = LAP
    A = ctx.convert_coo(rows, cols, I, J, V, dtype=np.float32)
    C = ctx.step1(A, A)
    for owner in (3, 1):
        ctx.set_option(pem.OPT_OWNER, owner)
        _refused(-2, ctx.step2, A, A, C)
    ctx.set_option(pem.OPT_OWNER, 0)
    ctx.step2(A, A, C)
    ctx.step3(A, A, C)
    oA = host.coo_to_csr(rows, cols, I, J, V)
    _assert_same(C, host.spgemm_f32(oA, oA))
    C.free()
    A.free()
    _clean_product(ctx)
    _assert_nothing_held(ctx)


def test_step3_on_dense_tiles_refused_then_retried(ctx):
    rows, cols, I, J, V = LAP
    A = ctx.convert_coo(rows, cols, I, J, V)
    assert A.info.nnz >= 8 * A.info.tiles
    C = ctx.step1(A, A)
    ctx.step2(A, A, C)                              # owner 0, dense tiles: no hit words
    ctx.set_option(pem.OPT_OWNER, 2)
    _refused(-2, ctx.step3, A, A, C)
    ctx.set_option(pem.OPT_OWNER, 0)
    ctx.step3(A, A, C)
    assert ctx.last_step3_kernel == 4
    _assert_same(C, host.spgemm_from_coo(rows, cols, I, J, V, False)[2])
    C.free()
    A.free()
    _clean_product(ctx)
    _assert_nothing_held(ctx)


@pytest.mark.parametrize("source", ["host", "device", "async"])
@pytest.mark.parametrize("flaw,code", [("duplicate", -4), ("out_of_range", -3)])
def test_convert_coo_refused(ctx, source, flaw, code):
    rows, cols, I, J, V = synth.random_sparse(300, 200, 3000, seed=5)
    I, J, V = np.array(I, np.int32), np.array(J, np.int32), np.array(V, np.float64)
    if flaw == "duplicate":
        I[-1], J[-1] = I[0], J[0]
    else:
        I[len(I) // 2] = rows
    if source == "device":
        import torch
        dI, dJ, dV = (torch.from_numpy(x).cuda() for x in (I, J, V))
        torch.cuda.synchronize()
        _refused(code, ctx.convert_coo, rows, cols, dI.data_ptr(), dJ.data_ptr(), dV.data_ptr(), False, len(I))
    else:
        ctx.set_option(pem.OPT_ASYNC_VALUES, int(source == "async"))
        _refused(code, ctx.convert_coo, rows, cols, I, J, V)
        ctx.set_option(pem.OPT_ASYNC_VALUES, 0)
    _clean_product(ctx)
    _assert_nothing_held(ctx)


def test_convert_csr_row_pointer_not_starting_at_zero(ctx):
    ptr = np.array([1, 2, 3], np.int32)
    _refused(-2, ctx.convert_csr, 2, 2, ptr, np.array([0, 1], np.int32), np.array([1.0, 2.0]))
    _clean_product(ctx)
    _assert_nothing_held(ctx)


@pytest.mark.parametrize("path", [1, 5])
def test_step1_shared_memory_refusal(ctx, path):
    A, B = hash_row_case(1025, 1 << 20)
    tA, tB = ctx.convert_coo(*A.coo()), ctx.convert_coo(*B.coo())
    ctx.set_option(pem.OPT_STEP1_PATH, path)
    _refused(-5, ctx.spgemm, tA, tB)
    ctx.set_option(pem.OPT_STEP1_PATH, 0)
    tA.free()
    tB.free()
    _clean_product(ctx)
    _assert_nothing_held(ctx)


def test_spgemm_fp32_under_owner_3(ctx):
    rows, cols, I, J, V = LAP
    A = ctx.convert_coo(rows, cols, I, J, V, dtype=np.float32)
    ctx.set_option(pem.OPT_OWNER, 3)
    _refused(-2, ctx.spgemm, A, A)
    ctx.set_option(pem.OPT_OWNER, 0)
    A.free()
    _clean_product(ctx)
    _assert_nothing_held(ctx)


def test_rectangular_a_times_a(ctx):
    A = ctx.convert_coo(*synth.random_sparse(90, 400, 2500, seed=3))
    _refused(-2, ctx.spgemm, A, A)
    A.free()
    _clean_product(ctx)
    _assert_nothing_held(ctx)
