"""Numeric-only re-multiplication against the full product, per config at full size:

  (a) steady-state pem_spgemm of the same operands (size plan and graph replayed, as bench.py times it)
  (b) pem_tiled_set_values from a device array, then pem_spgemm_numeric
  (c) the same from a pinned host array

    python tools/numeric_bench.py [--configs 1 2 3 4] [--steps 20] [--warmup 3] [--panels5 0]

(b) and (c) get new values on every step (seeded, different from the step before; written before the timed region).
Times are host clocks around calls that end in a device synchronisation; medians over the steps.  The refresh
kernel (k_refresh_vals) is timed with CUDA events on the engine's stream over `--steps` launches per operand, and
its rate is reported against its compulsory bytes (refresh_bytes).  A*A refreshes one handle; A*A^T refreshes A
and its device-built transpose with the same values.  At the end, (b)'s C is compared bit for bit with a full
product of the same values.  --panels5 N > 0 adds config 5 as N sequential tile-row panels, each (a) / (b) / (c)."""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import pem_spgemm_b200 as pem
from pem_spgemm_b200 import synth


def refresh_bytes(nnz, tiles, vsize, has_view):
    """Compulsory traffic of one k_refresh_vals launch: per nonzero the map entry (4 B), V (gathered) and vals; with
    the step-3 view also the (r, c) byte, the vals_t write and, per tile, its 16 column records (64 B); per tile the
    first-value offset (4 B)."""
    per_nnz = 4 + 2 * vsize + ((vsize + 1) if has_view else 0)
    per_tile = 4 + (64 if has_view else 0)
    return nnz * per_nnz + tiles * per_tile


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = (x.strip() for x in q.split(","))
        return name, power
    except Exception:
        return torch.cuda.get_device_name(), "unknown"


def median_ms(fn, steps, warmup):
    for i in range(warmup):
        fn(-1 - i)
    t = []
    for s in range(steps):
        t.append(fn(s))
    return float(np.median(t))


def run(ctx, name, A, B, panel, args, n, seed0):
    """One operand pair (B is A for A*A, A's transpose for A*A^T) and one panel (None: all of C)."""
    handles = [A] if B is A else [A, B]
    stream = torch.cuda.ExternalStream(ctx.stream)
    spg = (lambda: ctx.spgemm(A, B)) if panel is None else (lambda: ctx.spgemm(A, B, panel=panel))

    def full(_):
        t0 = time.perf_counter()
        C = spg()
        ms = (time.perf_counter() - t0) * 1e3
        C.free()
        return ms

    g = torch.Generator(device="cuda")
    dV = torch.empty(n, dtype=torch.float64, device="cuda")
    hV = torch.empty(n, dtype=torch.float64).pin_memory()
    C = spg()                                   # the result (b) and (c) refresh
    ms_a = median_ms(full, args.steps, args.warmup)
    r0 = ctx.graph_replays

    def new_values(step):
        g.manual_seed(seed0 + 1000 + step)
        dV.uniform_(-1, 1, generator=g)
        torch.cuda.synchronize()

    def numeric_dev(step):
        new_values(step)
        t0 = time.perf_counter()
        for T in handles:
            T.set_values(dV.data_ptr())
        ctx.spgemm_numeric(A, B, C)
        return (time.perf_counter() - t0) * 1e3

    def numeric_host(step):
        new_values(10000 + step)
        hV.copy_(dV)
        t0 = time.perf_counter()
        for T in handles:
            T.set_values(hV.numpy())
        ctx.spgemm_numeric(A, B, C)
        return (time.perf_counter() - t0) * 1e3

    ms_b = median_ms(numeric_dev, args.steps, args.warmup)
    s3 = ctx.kernel_ms()["step3_numeric"]
    ms_c = median_ms(numeric_host, args.steps, args.warmup)
    # refresh kernel alone: device V, events on the engine's stream around `steps` launches per handle
    kern = []
    for T in handles:
        i = T.info
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(stream)
        for _ in range(args.steps):
            T.set_values(dV.data_ptr())
        e1.record(stream)
        e1.synchronize()
        kms = e0.elapsed_time(e1) / args.steps
        by = refresh_bytes(i.nnz, i.tiles, 8, T is B)       # B's column-major view exists after the first product
        kern.append({"nnz": i.nnz, "tiles": i.tiles, "view": T is B, "ms": kms, "bytes": by, "GBps": by / kms / 1e6})
    # (b)'s C against a full product of the same values
    numeric_dev(12345)
    F = spg()
    same = np.array_equal(C.array("vals").view(np.uint64), F.array("vals").view(np.uint64)) and \
        np.array_equal(C.array("tile_nnz_ptr"), F.array("tile_nnz_ptr"))
    F.free()
    info = C.info
    C.free()
    return {"config": name, "panel": None if panel is None else [int(panel[0]), int(panel[1])], "C_nnz": info.nnz,
            "full_ms": ms_a, "numeric_dev_ms": ms_b, "numeric_host_ms": ms_c, "ratio_b_a": ms_b / ms_a,
            "step3_kernel": ctx.last_step3_kernel, "step3_kernel_ms": s3, "refresh": kern,
            "graph_replays_in_a": r0 > 0, "bit_identical": bool(same)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", type=int, nargs="+", default=[1, 2, 3, 4])
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--panels5", type=int, default=0)
    args = ap.parse_args()
    assert args.steps >= 10, "medians over at least 10 steps"
    if not torch.cuda.is_available():
        sys.exit("numeric_bench needs a CUDA device")
    name, power = card()
    print(json.dumps({"card": name, "power_limit": power}), flush=True)
    ok = True
    ctx = pem.Context(0)
    for k in args.configs + ([5] if args.panels5 > 0 else []):
        cname, tb, (rows, cols, I, J, V) = synth.config(k)
        A = ctx.convert_coo(rows, cols, I, J, V)
        B = ctx.transpose(A) if tb else A
        panels = [None]
        if k == 5:
            b = ctx.partition_panels(A, B, args.panels5)
            panels = [(b[q], b[q + 1]) for q in range(args.panels5)]
        for p in panels:
            r = run(ctx, cname, A, B, p, args, I.size, 100 * k)
            ok &= r["bit_identical"]
            print(json.dumps(r), flush=True)
        if B is not A:
            B.free()
        A.free()
        ctx.trim()
    ctx.close()
    if not ok:
        sys.exit("numeric_bench: a numeric product differs from the full product of the same values")


if __name__ == "__main__":
    main()
