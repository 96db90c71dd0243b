"""Sums of tiled matrices, per config at full size: S = alpha*A + beta*B with

  config 1: A - sigma*I   (I converted once; almost every tile of S is shared)
  config 2: A + A^T       (B the device transpose; partial overlap, power-law tile rows)
  config 3: A + A2        (A2 a second lp_like draw with another seed: rectangular, partial overlap)
  config 4: A + A^T       (the same pattern, the largest nnz)

  (a) Context.add (pem_tiled_add): wall ms, and device ms from CUDA events on the engine's stream around the call
  (b) the route that exists without it: a numpy union of the host COO the caller already holds (sorted keys, values
      rounded as in the contract), then convert_coo from host memory
  (c) Context.add_values (pem_tiled_add_values): device ms from CUDA events over repeated calls, with the compulsory
      bytes of its kernel (add_vals_bytes) and the rate they give

    python tools/add_bench.py [--configs 1 2 3 4] [--steps 20] [--warmup 3] [--host-steps 3]

Medians over the steps ((b) over --host-steps: it sorts every key on the host).  The card's name and power limit are
printed first, in the same run.  Each config ends with a bit-for-bit comparison of S from (a) with S from (b), every
array; the script exits non-zero on a mismatch."""
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

SIGMA = 0.75


def add_vals_bytes(nnz_s, tiles_s, nnz_a, tiles_a, nnz_b, tiles_b, vsize=8):
    """Compulsory traffic of k_add_vals when S has no column-major view: per nonzero of S its (r, c) byte read and its
    value written; every value of A and of B read once; per tile of S its value offset and its two source ids (12 B);
    per tile of A and of B its row masks, row pointers and value offset (52 B)."""
    return nnz_s * (1 + vsize) + (nnz_a + nnz_b) * vsize + tiles_s * 12 + (tiles_a + tiles_b) * 52


def host_union(a, b, alpha, beta):
    """The host route's union: (rows, cols, I, J, V) of alpha*a + beta*b, sorted by (row, col)."""
    rows, cols = a[0], a[1]
    ka = a[2].astype(np.int64) * cols + a[3]
    kb = b[2].astype(np.int64) * cols + b[3]
    keys = np.union1d(ka, kb)
    ia, ib = np.searchsorted(keys, ka), np.searchsorted(keys, kb)
    v = np.zeros(keys.size)
    in_b = np.zeros(keys.size, bool)
    in_b[ib] = True
    v[ib] = b[4] * beta
    pa = a[4] * alpha
    shared = in_b[ia]
    v[ia[~shared]] = pa[~shared]
    v[ia[shared]] = pa[shared] + v[ia[shared]]
    return rows, cols, (keys // cols).astype(np.int32), (keys % cols).astype(np.int32), v


def pair(k):
    """(name, A COO, B COO or "T" for the device transpose, alpha, beta)"""
    cname, _, a = synth.config(k)
    if k == 1:
        n = a[0]
        eye = (n, n, np.arange(n, dtype=np.int32), np.arange(n, dtype=np.int32), np.ones(n))
        return cname + ": A - sigma*I", a, eye, 1.0, -SIGMA
    if k == 3:
        return cname + ": A + A2", a, synth.lp_like(seed=4), 1.0, 1.0
    return cname + ": A + A^T", a, "T", 1.0, 1.0


def run(ctx, k, args):
    name, a, b, alpha, beta = pair(k)
    A = ctx.convert_coo(*a)
    if isinstance(b, str):
        B = ctx.transpose(A)
        b = (a[1], a[0], a[3], a[2], a[4])                 # the host COO a caller of A + A^T holds
    else:
        B = ctx.convert_coo(*b)
    stream = torch.cuda.ExternalStream(ctx.stream)
    S = ctx.add(A, B, alpha, beta)
    si, ai, bi = S.info, A.info, B.info
    out = {"config": name, "nnz_A": ai.nnz, "nnz_B": bi.nnz, "nnz_S": si.nnz, "tiles_S": si.tiles,
           "tiles_A": ai.tiles, "tiles_B": bi.tiles, "overlap_nnz": (ai.nnz + bi.nnz - si.nnz) / max(si.nnz, 1),
           "overlap_tiles": (ai.tiles + bi.tiles - si.tiles) / max(si.tiles, 1)}

    def add_wall(_):
        t0 = time.perf_counter()
        X = ctx.add(A, B, alpha, beta)
        ms = (time.perf_counter() - t0) * 1e3
        X.free()
        return ms

    out["add_ms"] = median_ms(add_wall, args.steps, args.warmup)
    spans = []
    for _ in range(args.steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        X = ctx.add(A, B, alpha, beta)
        e1.record(stream)
        e1.synchronize()
        spans.append(e0.elapsed_time(e1))
        X.free()
    out["add_device_ms"] = float(np.median(spans))

    def host_route(_):
        t0 = time.perf_counter()
        U = ctx.convert_coo(*host_union(a, b, alpha, beta))
        ms = (time.perf_counter() - t0) * 1e3
        U.free()
        return ms

    out["host_union_convert_ms"] = median_ms(host_route, args.host_steps, 1)
    out["ratio_a_b"] = out["add_ms"] / out["host_union_convert_ms"]

    # (c) add_values: events around batches of calls, new alpha each call
    reps = 10
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i in range(args.warmup):
        ctx.add_values(S, A, B, alpha + i, beta)
    ctx.sync()
    per = []
    for s in range(args.steps):
        e0.record(stream)
        for i in range(reps):
            ctx.add_values(S, A, B, alpha + 0.5 * i, beta)
        e1.record(stream)
        e1.synchronize()
        per.append(e0.elapsed_time(e1) / reps)
    ms = float(np.median(per))
    by = add_vals_bytes(si.nnz, si.tiles, ai.nnz, ai.tiles, bi.nnz, bi.tiles)
    out.update({"add_values_device_ms": ms, "add_values_bytes": by, "add_values_GBps": by / ms / 1e6})

    # S of (a) against S of (b), every array
    ctx.add_values(S, A, B, alpha, beta)
    U = ctx.convert_coo(*host_union(a, b, alpha, beta))
    same = all(np.array_equal(S.array(n).view(np.uint8), U.array(n).view(np.uint8)) for n in pem.T_ARRAYS)
    out["bit_identical"] = bool(same)
    for h in (U, S, B, A):
        h.free()
    ctx.trim()
    return out, same


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", type=int, nargs="+", default=[1, 2, 3, 4])
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--host-steps", type=int, default=3)
    args = ap.parse_args()
    assert args.steps >= 10, "medians over at least 10 steps"
    if not torch.cuda.is_available():
        sys.exit("add_bench needs a CUDA device")
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
        sys.exit("add_bench: a sum differs from the host union route")


if __name__ == "__main__":
    main()
