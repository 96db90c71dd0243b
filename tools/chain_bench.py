"""Results as operands, per config at full size: C = A*A (A*A^T for config 3), then the chained product T*A with
T = C.to_tiled().

  (a) Result.to_tiled (pem_result_to_tiled)
  (b) the route it replaces: Result.to_coo_device into device buffers, then convert_coo from those device pointers
  the chained product T*A: flop (pem_count_flop), nnz, steady-state time (size plan and graph replayed)
  numeric chain: A.set_values(dV); numeric(A, A, C); T.refresh_from(C); numeric(T, A, D)
  full chain:    C = A*A; T = C.to_tiled(); D = T*A (a new T every step: new size plans, no graph)

    python tools/chain_bench.py [--configs 1 2 3 4] [--steps 20] [--warmup 3] [--panels 1] [--max-flop 4e10]

Times are host clocks around calls that end in a device synchronisation; medians over the steps.  (a) is also timed
with CUDA events on the engine's stream around the call (its value copy, row count and scan, the two kernels of
operand.cu and the copy of the tile-row pointer), and its rate is reported against the call's compulsory bytes
(operand_bytes).  The chained product runs as --panels sequential tile-row panels of T; a config whose chained flop
exceeds --max-flop is skipped and reported as such.  At the end, the numeric chain's D is compared bit for bit with
the chain through (b); the script exits non-zero on a mismatch."""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import pem_spgemm_b200 as pem
from pem_spgemm_b200 import synth
from numeric_bench import card, median_ms


def operand_bytes(nnz, tiles, panel_rows, vsize):
    """Compulsory traffic of pem_result_to_tiled on a default-mode result: per nonzero the value read and written, the
    (r, c) byte and the value-map entry; per tile its row masks, tile row, tile column and offset read (48 B) and the
    masks, column masks, row pointers, occupancy words, tile indices and offset written (96 B); per matrix row of the
    panel its 8-byte position in C's row-major order, written once and read once."""
    return nnz * (2 * vsize + 1 + 4) + tiles * 144 + panel_rows * 16


def same_result(X, Y):
    return all(np.array_equal(X.array(n).view(np.uint8), Y.array(n).view(np.uint8))
               for n in ("row_ptr", "tile_col", "masks", "tile_nnz_ptr", "vals"))


def run(ctx, k, args):
    cname, tb, (rows, cols, I, J, V) = synth.config(k)
    A = ctx.convert_coo(rows, cols, I, J, V)
    B = ctx.transpose(A) if tb else A
    stream = torch.cuda.ExternalStream(ctx.stream)
    C = ctx.spgemm(A, B)
    ci = C.info
    out = {"config": cname, "product": "A*A^T" if tb else "A*A", "C_nnz": ci.nnz, "C_tiles": ci.tiles}

    def to_tiled(_):
        t0 = time.perf_counter()
        T = C.to_tiled()
        ms = (time.perf_counter() - t0) * 1e3
        T.free()
        return ms

    out["to_tiled_ms"] = median_ms(to_tiled, args.steps, args.warmup)
    spans = []
    for _ in range(args.steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        T = C.to_tiled()
        e1.record(stream)
        e1.synchronize()
        spans.append(e0.elapsed_time(e1))
        T.free()
    span = float(np.median(spans))
    by = operand_bytes(ci.nnz, ci.tiles, (ci.tile_row_end - ci.tile_row_begin) * 16, 8)
    out.update({"to_tiled_device_ms": span, "to_tiled_bytes": by, "to_tiled_GBps": by / span / 1e6})

    dr = torch.empty(max(ci.nnz, 1), dtype=torch.int32, device="cuda")
    dc = torch.empty_like(dr)
    dv = torch.empty(max(ci.nnz, 1), dtype=torch.float64, device="cuda")

    def via_coo():
        C.to_coo_device(dr.data_ptr(), dc.data_ptr(), dv.data_ptr())
        return ctx.convert_coo(ci.rows, ci.cols, dr.data_ptr(), dc.data_ptr(), dv.data_ptr(), nnz=ci.nnz)

    def export_convert(_):
        t0 = time.perf_counter()
        U = via_coo()
        ms = (time.perf_counter() - t0) * 1e3
        U.free()
        return ms

    out["export_convert_ms"] = median_ms(export_convert, args.steps, args.warmup)
    out["ratio_a_b"] = out["to_tiled_ms"] / out["export_convert_ms"]

    T = C.to_tiled()
    flop = ctx.count_flop(T, A)
    out["chained_flop"] = flop
    ok = True
    if flop > args.max_flop:
        out["chained"] = f"skipped: {flop:.3g} flop > --max-flop {args.max_flop:.3g}"
    else:
        b = ctx.partition_panels(T, A, args.panels)
        panels = [(int(b[q]), int(b[q + 1])) for q in range(args.panels)]

        def chained(_):
            t0 = time.perf_counter()
            for p in panels:
                ctx.spgemm(T, A, panel=p).free()
            return (time.perf_counter() - t0) * 1e3

        out["panels"] = args.panels
        out["chained_ms"] = median_ms(chained, args.steps, args.warmup)
        out["chained_GFLOPs"] = 2 * flop / out["chained_ms"] / 1e6
        g = torch.Generator(device="cuda")
        dV = torch.empty(I.size, dtype=torch.float64, device="cuda")
        Ds = []

        def new_values(step):
            g.manual_seed(1000 * k + step)
            dV.uniform_(-1, 1, generator=g)
            torch.cuda.synchronize()

        def numeric_chain(step):
            new_values(step)
            s = ctx.size_stalls
            t0 = time.perf_counter()
            for X in ([A] if B is A else [A, B]):
                X.set_values(dV.data_ptr())
            ctx.spgemm_numeric(A, B, C)
            T.refresh_from(C)
            for D in Ds:
                ctx.spgemm_numeric(T, A, D)
            ms = (time.perf_counter() - t0) * 1e3
            assert ctx.size_stalls == s, "the numeric chain stalled at a size read-back"
            return ms

        def full_chain(step):
            new_values(10000 + step)
            t0 = time.perf_counter()
            for X in ([A] if B is A else [A, B]):
                X.set_values(dV.data_ptr())
            C2 = ctx.spgemm(A, B)
            T2 = C2.to_tiled()
            C2.free()
            for p in panels:
                ctx.spgemm(T2, A, panel=p).free()
            T2.free()
            return (time.perf_counter() - t0) * 1e3

        # the full chain first: it holds no chained result of its own between steps, the numeric chain holds them all
        ctx.trim()
        out["full_chain_ms"] = median_ms(full_chain, args.steps, args.warmup)
        ctx.trim()
        Ds.extend(ctx.spgemm(T, A, panel=p) for p in panels)
        out["chained_nnz"] = sum(D.info.nnz for D in Ds)
        out["numeric_chain_ms"] = median_ms(numeric_chain, args.steps, args.warmup)
        out["ratio_numeric_full"] = out["numeric_chain_ms"] / out["full_chain_ms"]
        # the numeric chain's D against the chain through the export-and-convert route, same values
        numeric_chain(12345)
        U = via_coo()
        same = True
        for p, D in zip(panels, Ds):
            F = ctx.spgemm(U, A, panel=p)
            same &= same_result(D, F)
            F.free()
            D.free()
        U.free()
        out["bit_identical"] = bool(same)
        ok = same
    T.free()
    C.free()
    if B is not A:
        B.free()
    A.free()
    ctx.trim()
    return out, ok


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", type=int, nargs="+", default=[1, 2, 3, 4])
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--panels", type=int, default=1)
    ap.add_argument("--max-flop", type=float, default=4e10)
    args = ap.parse_args()
    assert args.steps >= 10, "medians over at least 10 steps"
    if not torch.cuda.is_available():
        sys.exit("chain_bench needs a CUDA device")
    name, power = card()
    print(json.dumps({"card": name, "power_limit": power}), flush=True)
    ok = True
    ctx = pem.Context(0)
    for k in args.configs:
        r, good = run(ctx, k, args)
        ok &= good
        print(json.dumps(r), flush=True)
    ctx.close()
    if not ok:
        sys.exit("chain_bench: a chained product differs from the chain through the export-and-convert route")


if __name__ == "__main__":
    main()
