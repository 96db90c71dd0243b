"""pem_spgemm_b200 — B200-native tiled SpGEMM engine (C = A^2, C = A*A^T, fp64, 16x16 tiles).

This package is a thin ctypes view of ``libpemspgemm.so`` (C ABI in ``include/pemspgemm.h``;
CUDA kernels in ``csrc/``).  The host-side mirror of the reference's process-level interface
(``pemspgemm <mtx> [0/1] [1]``, /root/reference/spgemm.cu:720-1568) is the C++ program in
``cli/``; Python is used for tests and the benchmark harness only.

There is no CPU fallback: importing works without a GPU (so the build can be checked), but
creating a :class:`Context` without a CUDA device or without the compiled library raises.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libpemspgemm.so")
CLI_PATH = os.path.join(_HERE, "bin", "pemspgemm")

PEM_OK = 0
STATUS = {0: "PEM_OK", -1: "PEM_ERR_CUDA", -2: "PEM_ERR_ARG", -3: "PEM_ERR_RANGE",
          -4: "PEM_ERR_DUPLICATE", -5: "PEM_ERR_LIMIT", -6: "PEM_ERR_NO_DEVICE", -7: "PEM_ERR_IO"}
OPT_KEEP_EMPTY_TILES = 1
OPT_STEP1_PATH = 2
OPT_OWNER = 3
OPT_S3_SMALL_NNZ = 4
OPT_S3_SMALL_PAIRS = 5
OPT_ASYNC_VALUES = 6
OPT_STEP2_KERNEL = 7
OPT_TRACE = 8
OPT_ESC_VARIANT = 9
OPT_CACHE_LIMIT_MB = 10
OPT_SIZE_PLANS = 11
OPT_GRAPHS = 12
OPT_GRAPH_LIMIT_MB = 13
OPT_POISON = 14                  # tests only: 0 or 0x100 | byte fills every allocated device block with that byte

# pem_tiled_array / pem_result_array -> (index, dtype)
T_ARRAYS = {
    "vals": (0, np.float64), "tile_nnz_ptr": (1, np.uint32), "masks": (2, np.uint16),
    "row_ptr": (3, np.uint8), "masks_t": (4, np.uint16), "tile_row_ptr": (5, np.int32),
    "tile_col_idx": (6, np.int32), "tile_row_idx": (7, np.int32), "col_occ": (8, np.uint16),
    "row_occ": (9, np.uint16), "row_col_idx": (10, np.uint8), "val_pos": (11, np.uint32),
}
R_ARRAYS = {
    "row_ptr": (0, np.int64), "tile_row": (1, np.int32), "tile_col": (2, np.int32),
    "pair_ptr": (3, np.int64), "pairs_a": (4, np.int32), "pairs_b": (5, np.int32),
    "masks": (6, np.uint16), "tile_nnz_ptr": (7, np.int64), "row_col_idx": (8, np.uint8),
    "vals": (9, np.float64),
}


class PemError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"{STATUS.get(code, code)}: {msg}")
        self.code = code


class Times(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("convert_kernel_ms", "convert_total_ms", "step1_ms", "step2_ms",
                                          "step3_ms", "kernel_ms", "total_ms", "malloc_ms")]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class TiledInfo(C.Structure):
    _fields_ = [("rows", C.c_int32), ("cols", C.c_int32), ("nnz", C.c_int64), ("tile_rows", C.c_int32),
                ("tile_cols", C.c_int32), ("tiles", C.c_int32)]


class ResultInfo(C.Structure):
    _fields_ = [("tile_row_begin", C.c_int32), ("tile_row_end", C.c_int32), ("rows", C.c_int32),
                ("cols", C.c_int32), ("tiles", C.c_int64), ("pairs", C.c_int64), ("nnz", C.c_int64),
                ("tile_products", C.c_int64)]


EXPORTS = [
    "pem_ctx_create", "pem_ctx_destroy", "pem_last_error", "pem_ctx_set_option", "pem_ctx_stream",
    "pem_ctx_sync", "pem_ctx_launch_count", "pem_ctx_last_sort_passes", "pem_ctx_kernel_ms", "pem_ctx_pool_mallocs", "pem_ctx_size_stalls", "pem_ctx_graph_replays", "pem_ctx_last_step3_kernel", "pem_ctx_pool_bytes", "pem_ctx_trim", "pem_convert_coo", "pem_convert_coo_f32", "pem_tiled_dtype", "pem_result_dtype", "pem_convert_csr", "pem_tiled_transpose",
    "pem_tiled_info_get", "pem_tiled_values_ready", "pem_tiled_set_values", "pem_tiled_set_values_f32", "pem_spgemm_numeric",
    "pem_tiled_free", "pem_tiled_get", "pem_tiled_device_ptr", "pem_count_flop", "pem_partition_panels",
    "pem_spgemm", "pem_spgemm_panel", "pem_step1_symbolic", "pem_step2_symbolic", "pem_step3_numeric",
    "pem_result_to_tiled", "pem_tiled_refresh_from_result", "pem_tiled_add", "pem_tiled_add_values",
    "pem_result_info_get", "pem_result_free", "pem_result_get", "pem_result_device_ptr",
    "pem_result_to_coo", "pem_result_to_coo_f32", "pem_result_to_csr", "pem_result_to_coo_device", "pem_result_checksum", "pem_mtx_read", "pem_mtx_write",
    "pem_free_host", "pem_write_lines_i32", "pem_write_lines_f64",
]

_lib = None


def build(verbose: bool = False) -> None:
    """Compile libpemspgemm.so and the CLI in-tree (nvcc, sm_100a)."""
    cmd = ["make", "-C", _HERE, "-j8", "all"]
    subprocess.check_call(cmd, stdout=None if verbose else subprocess.DEVNULL)


def load():
    """dlopen the engine; fail loudly if it was never built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    sig = {
        "pem_ctx_create": (C.c_int, [C.POINTER(vp), C.c_int]),
        "pem_ctx_destroy": (None, [vp]),
        "pem_last_error": (C.c_char_p, [vp]),
        "pem_ctx_set_option": (C.c_int, [vp, C.c_int, i64]),
        "pem_ctx_stream": (vp, [vp]),
        "pem_ctx_sync": (C.c_int, [vp]),
        "pem_ctx_launch_count": (i64, [vp]),
        "pem_ctx_last_sort_passes": (C.c_int, [vp]),
        "pem_ctx_pool_bytes": (i64, [vp]),
        "pem_ctx_trim": (C.c_int, [vp]),
        "pem_ctx_pool_mallocs": (i64, [vp]),
        "pem_ctx_size_stalls": (i64, [vp]),
        "pem_ctx_graph_replays": (i64, [vp]),
        "pem_ctx_last_step3_kernel": (C.c_int, [vp]),
        "pem_ctx_kernel_ms": (C.c_int, [vp, C.POINTER(C.c_double), C.c_int]),
        "pem_convert_coo": (C.c_int, [vp, i32, i32, i64, vp, vp, vp, C.c_int, C.POINTER(vp), C.POINTER(Times)]),
        "pem_convert_coo_f32": (C.c_int, [vp, i32, i32, i64, vp, vp, vp, C.c_int, C.POINTER(vp), C.POINTER(Times)]),
        "pem_tiled_dtype": (C.c_int, [vp]),
        "pem_result_dtype": (C.c_int, [vp]),
        "pem_result_to_coo_f32": (C.c_int, [vp, vp, vp, vp, vp]),
        "pem_convert_csr": (C.c_int, [vp, i32, i32, vp, vp, vp, C.c_int, C.POINTER(vp), C.POINTER(Times)]),
        "pem_tiled_transpose": (C.c_int, [vp, vp, C.POINTER(vp)]),
        "pem_tiled_info_get": (C.c_int, [vp, C.POINTER(TiledInfo)]),
        "pem_tiled_values_ready": (C.c_int, [vp, vp]),
        "pem_tiled_set_values": (C.c_int, [vp, vp, vp]),
        "pem_tiled_set_values_f32": (C.c_int, [vp, vp, vp]),
        "pem_spgemm_numeric": (C.c_int, [vp, vp, vp, vp, C.POINTER(Times)]),
        "pem_tiled_free": (None, [vp, vp]),
        "pem_tiled_get": (C.c_int, [vp, vp, C.c_int, vp, C.c_size_t]),
        "pem_tiled_device_ptr": (vp, [vp, C.c_int]),
        "pem_count_flop": (C.c_int, [vp, vp, vp, C.POINTER(C.c_uint64)]),
        "pem_partition_panels": (C.c_int, [vp, vp, vp, C.c_int, vp]),
        "pem_spgemm": (C.c_int, [vp, vp, vp, C.POINTER(vp), C.POINTER(Times)]),
        "pem_spgemm_panel": (C.c_int, [vp, vp, vp, i32, i32, C.POINTER(vp), C.POINTER(Times)]),
        "pem_step1_symbolic": (C.c_int, [vp, vp, vp, i32, i32, C.POINTER(vp)]),
        "pem_step2_symbolic": (C.c_int, [vp, vp, vp, vp]),
        "pem_step3_numeric": (C.c_int, [vp, vp, vp, vp]),
        "pem_result_to_tiled": (C.c_int, [vp, vp, C.POINTER(vp)]),
        "pem_tiled_refresh_from_result": (C.c_int, [vp, vp, vp]),
        "pem_tiled_add": (C.c_int, [vp, C.c_double, vp, C.c_double, vp, C.POINTER(vp)]),
        "pem_tiled_add_values": (C.c_int, [vp, vp, C.c_double, vp, C.c_double, vp]),
        "pem_result_info_get": (C.c_int, [vp, C.POINTER(ResultInfo)]),
        "pem_result_free": (None, [vp, vp]),
        "pem_result_get": (C.c_int, [vp, vp, C.c_int, vp, C.c_size_t]),
        "pem_result_device_ptr": (vp, [vp, C.c_int]),
        "pem_result_to_coo": (C.c_int, [vp, vp, vp, vp, vp]),
        "pem_result_to_csr": (C.c_int, [vp, vp, vp, vp, vp]),
        "pem_result_to_coo_device": (C.c_int, [vp, vp, vp, vp, vp, vp]),
        "pem_result_checksum": (C.c_int, [vp, vp, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
        "pem_mtx_read": (C.c_int, [C.c_char_p, C.POINTER(i32), C.POINTER(i32), C.POINTER(i64), C.POINTER(vp),
                                   C.POINTER(vp), C.POINTER(vp), C.POINTER(C.c_int), C.c_char_p, C.c_size_t]),
        "pem_mtx_write": (C.c_int, [C.c_char_p, i32, i32, i64, vp, vp, vp]),
        "pem_write_lines_i32": (C.c_int, [C.c_char_p, vp, i64, C.c_int]),
        "pem_write_lines_f64": (C.c_int, [C.c_char_p, vp, i64, C.c_int]),
        "pem_free_host": (None, [vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def _ptr(a):
    """Host numpy array or raw device pointer (int) -> void*."""
    if a is None:
        return None
    if isinstance(a, (int, np.integer)):
        return C.c_void_p(int(a))
    return a.ctypes.data_as(C.c_void_p)


class Context:
    """One engine context (stream + memory pool) on one GPU."""

    def __init__(self, device: int = 0):
        L = load()
        h = C.c_void_p()
        rc = L.pem_ctx_create(C.byref(h), device)
        if rc != PEM_OK:
            raise PemError(rc, "pem_ctx_create failed (no CUDA device? there is no CPU fallback)")
        self._h = h
        self.device = device

    def _check(self, rc: int):
        if rc != PEM_OK:
            raise PemError(rc, load().pem_last_error(self._h).decode())

    def close(self):
        if getattr(self, "_h", None):
            load().pem_ctx_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def set_option(self, option: int, value: int):
        self._check(load().pem_ctx_set_option(self._h, option, value))

    @property
    def stream(self) -> int:
        return int(load().pem_ctx_stream(self._h) or 0)

    def sync(self):
        self._check(load().pem_ctx_sync(self._h))

    @property
    def launch_count(self) -> int:
        return int(load().pem_ctx_launch_count(self._h))

    @property
    def last_sort_passes(self) -> int:
        return int(load().pem_ctx_last_sort_passes(self._h))

    def kernel_ms(self) -> dict:
        """Device time of the individually timed kernels of the last spgemm call (CUDA events)."""
        a = (C.c_double * 4)()
        load().pem_ctx_kernel_ms(self._h, a, 4)
        return {"k_expand": a[0], "radix_sort": a[1], "k_step2_pairs": a[2], "step3_numeric": a[3]}

    @property
    def pool_mallocs(self) -> int:
        return int(load().pem_ctx_pool_mallocs(self._h))

    @property
    def last_step3_kernel(self) -> int:
        return int(load().pem_ctx_last_step3_kernel(self._h))

    @property
    def size_stalls(self) -> int:
        """Host stalls at device-size read-backs inside products since the context was created."""
        return int(load().pem_ctx_size_stalls(self._h))

    @property
    def graph_replays(self) -> int:
        """Products that ran as one CUDA-graph launch since the context was created (OPT_GRAPHS)."""
        return int(load().pem_ctx_graph_replays(self._h))

    def trim(self):
        """Hand the cached device blocks back to the driver."""
        self._check(load().pem_ctx_trim(self._h))

    @property
    def pool_bytes(self) -> int:
        return int(load().pem_ctx_pool_bytes(self._h))

    # -- conversion -----------------------------------------------------------------------
    def convert_coo(self, rows, cols, I, J, V, transpose=False, nnz=None, times: Times | None = None,
                    dtype=np.float64) -> "Tiled":
        """COO -> tiled CSR.  I/J/V are numpy arrays (host) or integer device pointers
        (then ``nnz`` is required).  ``dtype`` float64 (default) or float32 selects the value type."""
        f32 = np.dtype(dtype) == np.float32
        if not isinstance(I, (int, np.integer)):
            I = np.ascontiguousarray(I, np.int32); J = np.ascontiguousarray(J, np.int32)
            V = np.ascontiguousarray(V, np.float32 if f32 else np.float64)
            nnz = I.size
        h = C.c_void_p()
        self._keep = (I, J, V)
        fn = load().pem_convert_coo_f32 if f32 else load().pem_convert_coo
        rc = fn(self._h, rows, cols, nnz, _ptr(I), _ptr(J), _ptr(V), int(bool(transpose)),
                C.byref(h), C.byref(times) if times is not None else None)
        self._keep = None
        self._check(rc)
        return Tiled(self, h)

    def convert_csr(self, rows, cols, row_ptr, col_idx, vals, transpose=False, times: Times | None = None) -> "Tiled":
        """CSR -> tiled CSR.  Arrays are numpy (host) or integer device pointers (all three alike)."""
        if not isinstance(row_ptr, (int, np.integer)):
            row_ptr = np.ascontiguousarray(row_ptr, np.int32); col_idx = np.ascontiguousarray(col_idx, np.int32)
            vals = np.ascontiguousarray(vals, np.float64)
        h = C.c_void_p()
        rc = load().pem_convert_csr(self._h, rows, cols, _ptr(row_ptr), _ptr(col_idx), _ptr(vals), int(bool(transpose)),
                                    C.byref(h), C.byref(times) if times is not None else None)
        self._check(rc)
        return Tiled(self, h)

    def transpose(self, A: "Tiled") -> "Tiled":
        """A^T from A's tiles, on the device."""
        h = C.c_void_p()
        self._check(load().pem_tiled_transpose(self._h, A._h, C.byref(h)))
        return Tiled(self, h)

    def count_flop(self, A: "Tiled", B: "Tiled") -> int:
        f = C.c_uint64()
        self._check(load().pem_count_flop(self._h, A._h, B._h, C.byref(f)))
        return int(f.value)

    def partition_panels(self, A: "Tiled", B: "Tiled", nparts: int) -> np.ndarray:
        b = np.zeros(nparts + 1, np.int32)
        self._check(load().pem_partition_panels(self._h, A._h, B._h, nparts, _ptr(b)))
        return b

    # -- sums -----------------------------------------------------------------------------
    def add(self, A: "Tiled", B: "Tiled", alpha: float = 1.0, beta: float = 1.0) -> "Tiled":
        """S = alpha*A + beta*B as a new tiled matrix on the union of the patterns (nothing dropped, no fused
        multiply-add); A and B may be freed after."""
        h = C.c_void_p()
        self._check(load().pem_tiled_add(self._h, float(alpha), A._h, float(beta), B._h, C.byref(h)))
        return Tiled(self, h)

    def add_values(self, S: "Tiled", A: "Tiled", B: "Tiled", alpha: float = 1.0, beta: float = 1.0):
        """Recompute S = alpha*A + beta*B in place from the current values of A and B, the handles S was built from by
        ``add``, in that order."""
        self._check(load().pem_tiled_add_values(self._h, S._h, float(alpha), A._h, float(beta), B._h))

    # -- SpGEMM ---------------------------------------------------------------------------
    def spgemm(self, A: "Tiled", B: "Tiled", times: Times | None = None, panel=None) -> "Result":
        h = C.c_void_p()
        t = C.byref(times) if times is not None else None
        if panel is None:
            rc = load().pem_spgemm(self._h, A._h, B._h, C.byref(h), t)
        else:
            rc = load().pem_spgemm_panel(self._h, A._h, B._h, int(panel[0]), int(panel[1]), C.byref(h), t)
        self._check(rc)
        return Result(self, h)

    def spgemm_numeric(self, A: "Tiled", B: "Tiled", Cr: "Result", times: Times | None = None):
        """Recompute Cr's values in place from the current values of A and B (the handles Cr was computed from),
        on Cr's structure: step 3 only, the kernel Cr was built with."""
        self._check(load().pem_spgemm_numeric(self._h, A._h, B._h, Cr._h, C.byref(times) if times is not None else None))

    def step1(self, A: "Tiled", B: "Tiled", panel=None) -> "Result":
        h = C.c_void_p()
        rb, re = (0, A.info.tile_rows) if panel is None else panel
        self._check(load().pem_step1_symbolic(self._h, A._h, B._h, int(rb), int(re), C.byref(h)))
        return Result(self, h)

    def step2(self, A: "Tiled", B: "Tiled", Cr: "Result"):
        self._check(load().pem_step2_symbolic(self._h, A._h, B._h, Cr._h))

    def step3(self, A: "Tiled", B: "Tiled", Cr: "Result"):
        self._check(load().pem_step3_numeric(self._h, A._h, B._h, Cr._h))


class Tiled:
    def __init__(self, ctx: Context, h):
        self.ctx, self._h = ctx, h

    @property
    def info(self) -> TiledInfo:
        i = TiledInfo()
        load().pem_tiled_info_get(self._h, C.byref(i))
        return i

    @property
    def dtype(self):
        return np.float32 if load().pem_tiled_dtype(self._h) == 1 else np.float64

    def array(self, name: str) -> np.ndarray:
        idx, dt = T_ARRAYS[name]
        if name == "vals":
            dt = self.dtype
        i = self.info
        n = {"vals": i.nnz, "tile_nnz_ptr": i.tiles + 1, "masks": i.tiles * 16, "row_ptr": i.tiles * 16,
             "masks_t": i.tiles * 16, "tile_row_ptr": i.tile_rows + 1, "tile_col_idx": i.tiles,
             "tile_row_idx": i.tiles, "col_occ": i.tiles, "row_occ": i.tiles, "row_col_idx": i.nnz,
             "val_pos": i.nnz}[name]
        out = np.empty(n, dt)
        self.ctx._check(load().pem_tiled_get(self.ctx._h, self._h, idx, _ptr(out), out.nbytes))
        return out

    def set_values(self, V):
        """New values on the same pattern, in place: V is a numpy array (host) or an integer device pointer, nnz
        entries in the order of the input this matrix was converted from (for a transpose: its source's input),
        fp32 or fp64 by the matrix's dtype.  A device V is read in the context's stream order."""
        f32 = self.dtype == np.float32
        if V is not None and not isinstance(V, (int, np.integer)):
            V = np.ascontiguousarray(V, np.float32 if f32 else np.float64)
            if V.size != self.info.nnz:
                raise ValueError(f"set_values: {V.size} values for a matrix with {self.info.nnz} nonzeros")
        fn = load().pem_tiled_set_values_f32 if f32 else load().pem_tiled_set_values
        self.ctx._check(fn(self.ctx._h, self._h, _ptr(V)))

    def refresh_from(self, result: "Result"):
        """Write ``result``'s current values into this matrix in place; it must have been built by
        ``Result.to_tiled`` from a result of the same product and panel (e.g. after ``Context.spgemm_numeric``)."""
        self.ctx._check(load().pem_tiled_refresh_from_result(self.ctx._h, self._h, result._h))

    def values_ready(self):
        """Block until the engine no longer reads the host value array this matrix was converted from."""
        self.ctx._check(load().pem_tiled_values_ready(self.ctx._h, self._h))

    def free(self):
        if self._h:
            load().pem_tiled_free(self.ctx._h, self._h)
            self._h = None


class Result:
    def __init__(self, ctx: Context, h):
        self.ctx, self._h = ctx, h

    @property
    def info(self) -> ResultInfo:
        i = ResultInfo()
        load().pem_result_info_get(self._h, C.byref(i))
        return i

    @property
    def dtype(self):
        return np.float32 if load().pem_result_dtype(self._h) == 1 else np.float64

    def array(self, name: str) -> np.ndarray:
        idx, dt = R_ARRAYS[name]
        if name == "vals":
            dt = self.dtype
        i = self.info
        n = {"row_ptr": i.tile_row_end - i.tile_row_begin + 1, "tile_row": i.tiles, "tile_col": i.tiles,
             "pair_ptr": i.tiles + 1, "pairs_a": i.pairs, "pairs_b": i.pairs, "masks": i.tiles * 16,
             "tile_nnz_ptr": i.tiles + 1, "row_col_idx": i.nnz, "vals": i.nnz}[name]
        out = np.empty(n, dt)
        self.ctx._check(load().pem_result_get(self.ctx._h, self._h, idx, _ptr(out), out.nbytes))
        return out

    def to_coo(self, values: bool = True):
        """(rows, cols, vals) on the host, sorted by (row, col)."""
        n = self.info.nnz
        r = np.empty(n, np.int32); c = np.empty(n, np.int32)
        f32 = self.dtype == np.float32
        v = np.empty(n, self.dtype) if values else None
        fn = load().pem_result_to_coo_f32 if f32 else load().pem_result_to_coo
        self.ctx._check(fn(self.ctx._h, self._h, _ptr(r), _ptr(c), _ptr(v)))
        return r, c, v

    def to_csr(self):
        """(row_ptr int64, cols, vals) on the host, ascending columns inside a row."""
        i = self.info
        nrows = max(0, min(i.rows, i.tile_row_end * 16) - i.tile_row_begin * 16)
        rp = np.empty(nrows + 1, np.int64); c = np.empty(i.nnz, np.int32); v = np.empty(i.nnz, np.float64)
        self.ctx._check(load().pem_result_to_csr(self.ctx._h, self._h, _ptr(rp), _ptr(c), _ptr(v)))
        return rp, c, v

    def to_coo_into(self, rows_ptr, cols_ptr, vals_ptr):
        """Same, into caller-owned HOST buffers given as integer addresses (pinned memory for full PCIe
        speed); each must hold ``info.nnz`` entries; 0 skips an array."""
        self.ctx._check(load().pem_result_to_coo(self.ctx._h, self._h, C.c_void_p(rows_ptr or None),
                                                 C.c_void_p(cols_ptr or None), C.c_void_p(vals_ptr or None)))

    def to_coo_device(self, rows_ptr, cols_ptr, vals_ptr, row_ptr_ptr=0):
        """Same, into caller-owned DEVICE buffers given as integer addresses: ``info.nnz`` rows / cols / vals (fp32
        values for an fp32 result) and, when ``row_ptr_ptr`` is given, the CSR row pointer of the result's tile rows,
        int64 [(tile_row_end - tile_row_begin) * 16 + 1]; 0 skips an array."""
        self.ctx._check(load().pem_result_to_coo_device(self.ctx._h, self._h, C.c_void_p(rows_ptr or None),
                                                        C.c_void_p(cols_ptr or None), C.c_void_p(vals_ptr or None),
                                                        C.c_void_p(row_ptr_ptr or None)))

    def to_tiled(self) -> Tiled:
        """This result as a new, independent tiled matrix (the next operand of a chain of products): the arrays
        ``convert_coo(*self.to_coo())`` would build, C's full shape for a panel.  The result may be freed after."""
        h = C.c_void_p()
        self.ctx._check(load().pem_result_to_tiled(self.ctx._h, self._h, C.byref(h)))
        return Tiled(self.ctx, h)

    def checksum(self):
        s, a = C.c_double(), C.c_double()
        self.ctx._check(load().pem_result_checksum(self.ctx._h, self._h, C.byref(s), C.byref(a)))
        return s.value, a.value

    def free(self):
        if self._h:
            load().pem_result_free(self.ctx._h, self._h)
            self._h = None


def mtx_write(path: str, rows: int, cols: int, I, J, V) -> None:
    I = np.ascontiguousarray(I, np.int32); J = np.ascontiguousarray(J, np.int32)
    V = np.ascontiguousarray(V, np.float64)
    rc = load().pem_mtx_write(path.encode(), rows, cols, I.size, _ptr(I), _ptr(J), _ptr(V))
    if rc != PEM_OK:
        raise PemError(rc, f"cannot write {path}")


def write_lines(path: str, x, append: bool = False) -> None:
    """One number per line, the format of the reference's COO dump files (int32 as is, float64 fixed with 17 decimals)."""
    x = np.ascontiguousarray(x)
    if x.dtype == np.float64:
        rc = load().pem_write_lines_f64(path.encode(), _ptr(x), x.size, int(append))
    else:
        x = np.ascontiguousarray(x, np.int32)
        rc = load().pem_write_lines_i32(path.encode(), _ptr(x), x.size, int(append))
    if rc != PEM_OK:
        raise PemError(rc, f"cannot write {path}")


def mtx_read(path: str):
    """-> (rows, cols, I, J, V, is_symmetric)"""
    L = load()
    rows, cols, nnz, sym = C.c_int32(), C.c_int32(), C.c_int64(), C.c_int()
    pi, pj, pv = C.c_void_p(), C.c_void_p(), C.c_void_p()
    err = C.create_string_buffer(256)
    rc = L.pem_mtx_read(path.encode(), C.byref(rows), C.byref(cols), C.byref(nnz), C.byref(pi), C.byref(pj),
                        C.byref(pv), C.byref(sym), err, 256)
    if rc != PEM_OK:
        raise PemError(rc, err.value.decode())
    n = nnz.value
    try:
        I = np.ctypeslib.as_array(C.cast(pi, C.POINTER(C.c_int32)), (n,)).copy() if n else np.zeros(0, np.int32)
        J = np.ctypeslib.as_array(C.cast(pj, C.POINTER(C.c_int32)), (n,)).copy() if n else np.zeros(0, np.int32)
        V = np.ctypeslib.as_array(C.cast(pv, C.POINTER(C.c_double)), (n,)).copy() if n else np.zeros(0)
    finally:
        L.pem_free_host(pi); L.pem_free_host(pj); L.pem_free_host(pv)
    return rows.value, cols.value, I, J, V, bool(sym.value)
