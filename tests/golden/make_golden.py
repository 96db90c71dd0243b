"""Generates the golden fixtures in this directory by running the UNMODIFIED reference
(/root/reference/spgemm.cu rebuilt for sm_100 as oracle/_ref/pemspgemm_ref, see oracle/Makefile)
on a B200 through its own CLI and collecting its COO dump (/tmp/SPGEMM_RESULT_*.txt,
spgemm.cu:1527-1560) and its report.

    gpurun -- python tests/golden/make_golden.py        # writes gpurun_out/golden/*.npz
    gpurun -- python tests/golden/make_golden.py --bin pemspgemm_ref61 --timeout 120 rand300k_a2 lap600_a2 webbase270k_a2
    cp gpurun_out/golden/*.npz tests/golden/            # commit

`--bin` picks the rebuild under oracle/_ref (pemspgemm_ref = compute_100 PTX; pemspgemm_ref61 = the
reference's own compute_61 PTX, /root/reference/Makefile:13); case names select a subset.

The inputs are re-created from pem_spgemm_b200.synth by name and seed (CASES below), so only the
reference's OUTPUT is stored.  The reference never zeroes Ctiles_vals (SURVEY.md section 4 quirk 1);
a dump whose values are not finite is recorded as such rather than "fixed".
"""
import os
import re
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import pem_spgemm_b200 as pem           # noqa: E402  (only its Matrix Market writer is used)
from pem_spgemm_b200 import synth       # noqa: E402

CASES = {
    # name: (generator call, transpose_b)
    "lap32_a2": (lambda: synth.laplacian2d(32), False),
    "rand300_a2": (lambda: synth.random_sparse(300, 300, 3000, seed=2), False),
    "rand120x700_aat": (lambda: synth.random_sparse(120, 700, 3000, seed=7), True),
    "cage8_a2": (lambda: synth.cage_like(8, 9, 9), False),
    "webbase_small_a2": (lambda: synth.config(2, small=True)[2], False),
    "lap256_a2": (lambda: synth.laplacian2d(256), False),       # config 1 at full size
    # more than 16,384 B tile columns: the reference's NSPARSE hash step 1 (spgemm.cu:1142)
    "rand300k_a2": (lambda: synth.random_sparse(300_000, 300_000, 60_000, seed=5), False),
    "lap600_a2": (lambda: synth.laplacian2d(600), False),
    "webbase270k_a2": (lambda: synth.webbase_like(n=270_007, target_nnz=800_000, max_deg=2000), False),
}
SUMMARY_ONLY = {"lap256_a2", "lap600_a2", "webbase270k_a2"}   # keep only counts, checksums and a structure hash for the larger ones
# summary plus this many entries of the dump, for fixtures whose full COO would exceed 1 MB
SAMPLED = {"webbase_small_a2": 16_384}


def sample(r, c, v, k):
    """A seeded sample of k dump entries: their positions in the (row, col)-sorted COO and the entries."""
    p = np.sort(np.random.default_rng(0).choice(r.size, min(k, r.size), replace=False)).astype(np.int32)
    return dict(sample_pos=p, rows_s=r[p], cols_s=c[p], vals_s=v[p])


def struct_hash(r, c):
    """Order-independent 64-bit digest of the (row, col) set."""
    x = (r.astype(np.uint64) << np.uint64(32)) | c.astype(np.uint64)
    x ^= x >> np.uint64(33)
    x *= np.uint64(0xFF51AFD7ED558CCD)
    x ^= x >> np.uint64(29)
    return int(x.sum(dtype=np.uint64))


def main():
    import argparse
    ap = argparse.ArgumentParser()
    ap.add_argument("--bin", default="pemspgemm_ref")
    ap.add_argument("--timeout", type=int, default=600)
    ap.add_argument("cases", nargs="*")
    args = ap.parse_args()
    ref = os.path.join(ROOT, "oracle", "_ref", args.bin)
    out_dir = os.path.join(ROOT, "gpurun_out", "golden")
    os.makedirs(out_dir, exist_ok=True)
    work = "/tmp/pem_golden"
    os.makedirs(work, exist_ok=True)
    for name, (gen, tb) in CASES.items():
        if args.cases and name not in args.cases:
            continue
        rows, cols, I, J, V = gen()
        mtx = os.path.join(work, name + ".mtx")
        pem.mtx_write(mtx, rows, cols, I, J, V)
        for f in ("NNZ", "ROWS", "COLS", "VALS"):
            try:
                os.remove(f"/tmp/SPGEMM_RESULT_{f}.txt")
            except FileNotFoundError:
                pass
        try:
            p = subprocess.run([ref, mtx, "1"] + (["1"] if tb else []), cwd=work, capture_output=True, text=True, timeout=args.timeout)
        except subprocess.TimeoutExpired as e:
            print(name, "TIMEOUT after", args.timeout, "s; stdout tail:", (e.stdout or b"")[-400:], flush=True)
            continue
        print(name, "rc", p.returncode, flush=True)
        if p.returncode != 0:
            print(p.stdout[-2000:], p.stderr[-2000:])
            continue
        rep = p.stdout
        nnz = int(open("/tmp/SPGEMM_RESULT_NNZ.txt").read())
        r = np.loadtxt("/tmp/SPGEMM_RESULT_ROWS.txt", dtype=np.int64, ndmin=1).astype(np.int32)
        c = np.loadtxt("/tmp/SPGEMM_RESULT_COLS.txt", dtype=np.int64, ndmin=1).astype(np.int32)
        v = np.loadtxt("/tmp/SPGEMM_RESULT_VALS.txt", dtype=np.float64, ndmin=1)
        assert r.size == nnz == c.size == v.size
        meta = dict(
            c_tiles=int(re.search(r"C tiles: (\d+)", rep).group(1)),
            c_nnz=int(re.search(r"C nnz: (\d+)", rep).group(1)),
            flop=int(re.search(r"Flop count: (\d+)", rep).group(1)),
            step1_path="NSPARSE" if "step1 using NSPARSE" in rep else "SPA",
            transpose_b=int(tb), rows=rows, cols=cols, nnz_a=int(I.size),
            val_sum=float(v.sum()), val_abs_sum=float(np.abs(v).sum()),
            struct_hash=np.uint64(struct_hash(r, c)), ref_bin=args.bin,
        )
        print(meta, flush=True)
        if name in SUMMARY_ONLY:
            np.savez_compressed(os.path.join(out_dir, name + ".npz"), **{k: np.array(x) for k, x in meta.items()})
        elif name in SAMPLED:
            np.savez_compressed(os.path.join(out_dir, name + ".npz"), **sample(r, c, v, SAMPLED[name]),
                                **{k: np.array(x) for k, x in meta.items()})
        else:
            np.savez_compressed(os.path.join(out_dir, name + ".npz"), rows_c=r, cols_c=c, vals_c=v,
                                **{k: np.array(x) for k, x in meta.items()})


if __name__ == "__main__":
    main()
