"""Pins: the host oracle (CPU) and the CUDA engine (GPU) against dumps of the reference's own
sm_100 rebuild run on a B200 (tests/golden/README.md)."""
import glob
import os

import numpy as np
import pytest

from oracle import host
from pem_spgemm_b200 import synth

HERE = os.path.dirname(os.path.abspath(__file__))
CASES = {
    "lap32_a2": (lambda: synth.laplacian2d(32), False),
    "rand300_a2": (lambda: synth.random_sparse(300, 300, 3000, seed=2), False),
    "rand120x700_aat": (lambda: synth.random_sparse(120, 700, 3000, seed=7), True),
    "cage8_a2": (lambda: synth.cage_like(8, 9, 9), False),
    "webbase_small_a2": (lambda: synth.config(2, small=True)[2], False),
    "lap256_a2": (lambda: synth.laplacian2d(256), False),
    # the reference's NSPARSE hash step 1 (> 16,384 B tile columns, spgemm.cu:1142); produced by the
    # compute_61-PTX rebuild oracle/_ref/pemspgemm_ref61 (the compute_100 one does not terminate there)
    "rand300k_a2": (lambda: synth.random_sparse(300_000, 300_000, 60_000, seed=5), False),
    "lap600_a2": (lambda: synth.laplacian2d(600), False),
    "webbase270k_a2": (lambda: synth.webbase_like(n=270_007, target_nnz=800_000, max_deg=2000), False),
}


def struct_hash(r, c):
    """Order-independent 64-bit digest of the (row, col) set (same as tests/golden/make_golden.py)."""
    x = (r.astype(np.uint64) << np.uint64(32)) | c.astype(np.uint64)
    x ^= x >> np.uint64(33)
    x *= np.uint64(0xFF51AFD7ED558CCD)
    x ^= x >> np.uint64(29)
    return int(x.sum(dtype=np.uint64))


def _load(name):
    return np.load(os.path.join(HERE, "golden", name + ".npz"))


def _check_sample(g, r, c, v):
    """Fixtures too large to store whole keep a seeded sample of the dump's entries (make_golden.sample)."""
    if "sample_pos" in g:
        p = g["sample_pos"]
        assert np.array_equal(r[p], g["rows_s"]) and np.array_equal(c[p], g["cols_s"])
        np.testing.assert_allclose(v[p], g["vals_s"], rtol=1e-12, atol=1e-16)


def test_every_fixture_has_a_case():
    names = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(HERE, "golden", "*.npz")))
    assert names == sorted(CASES)


@pytest.mark.parametrize("name", sorted(CASES))
def test_oracle_matches_reference_dump(name):
    gen, tb = CASES[name]
    g = _load(name)
    rows, cols, I, J, V = gen()
    assert I.size == int(g["nnz_a"]) and rows == int(g["rows"]) and int(g["transpose_b"]) == int(tb)
    A, B, C = host.spgemm_from_coo(rows, cols, I, J, V, tb)
    assert host.flop(A, B) == int(g["flop"])
    assert C.nnz == int(g["c_nnz"])
    np.testing.assert_allclose([C.val.sum(), np.abs(C.val).sum()], [float(g["val_sum"]), float(g["val_abs_sum"])],
                               rtol=1e-11)
    if "rows_c" in g:
        r, c, v = C.to_coo()
        assert np.array_equal(r, g["rows_c"]) and np.array_equal(c, g["cols_c"])
        np.testing.assert_allclose(v, g["vals_c"], rtol=1e-12, atol=1e-16)
    elif "struct_hash" in g:
        r, c, v = C.to_coo()
        assert struct_hash(r, c) == int(g["struct_hash"])
        _check_sample(g, r, c, v)


def test_nsparse_path_fixtures_present():
    """At least one fixture must come from the reference's NSPARSE step-1 path."""
    assert any(str(_load(n)["step1_path"]) == "NSPARSE" for n in CASES)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_engine_matches_reference_dump(engine, name):
    import pem_spgemm_b200 as pem
    gen, tb = CASES[name]
    g = _load(name)
    rows, cols, I, J, V = gen()
    A = engine.convert_coo(rows, cols, I, J, V)
    B = engine.convert_coo(rows, cols, I, J, V, transpose=True) if tb else A
    assert engine.count_flop(A, B) == int(g["flop"])
    engine.set_option(pem.OPT_KEEP_EMPTY_TILES, 1)      # "C tiles" as the reference counts them
    try:
        C = engine.spgemm(A, B)
    finally:
        engine.set_option(pem.OPT_KEEP_EMPTY_TILES, 0)
    assert (C.info.tiles, C.info.nnz) == (int(g["c_tiles"]), int(g["c_nnz"]))
    C.free()
    C = engine.spgemm(A, B)
    assert C.info.nnz == int(g["c_nnz"])
    if "rows_c" in g:
        r, c, v = C.to_coo()
        assert np.array_equal(r, g["rows_c"]) and np.array_equal(c, g["cols_c"])
        np.testing.assert_allclose(v, g["vals_c"], rtol=1e-12, atol=1e-16)
    elif "struct_hash" in g:
        r, c, v = C.to_coo()
        assert struct_hash(r, c) == int(g["struct_hash"])
        np.testing.assert_allclose([v.sum(), np.abs(v).sum()], [float(g["val_sum"]), float(g["val_abs_sum"])], rtol=1e-11)
        _check_sample(g, r, c, v)
    C.free()
    if B is not A:
        B.free()
    A.free()
