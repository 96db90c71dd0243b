#!/usr/bin/env python
"""Benchmark of the SpGEMM hot path: SpGEMM GFLOP/s = 2*flop / time for C = A^2 (or A*A^T).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config 1..5] [--impl ours|reference] [--dump-outputs DIR]

One "step" is one full SpGEMM (steps 1-3 including allocation, i.e. one iteration of the
reference's timed loop, /root/reference/spgemm.cu:1133-1357) on operands already resident in HBM
in tiled form.  At N > 1 (torchrun, one process per GPU) A's tile rows are split into N
flop-balanced panels, B is replicated, each rank multiplies its panel, and the per-shard
{nnz, tiles, pairs} are all-gathered over NCCL (the only exchange on this path); the time is the
max over ranks and the value is the whole job's 2*flop / time ("strong" scaling: same matrix at
every N).  Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CONFIG_TEXT = {
    1: "config1: A^2, 2-D 5-point Laplacian 256x256 grid (n=65,536)",
    2: "config2: A^2, synthetic webbase-1M-shaped power-law matrix (n=1,000,005, nnz=3,091,482)",
    3: "config3: A*A^T, synthetic LP-shaped 100,000 x 1,000,000, 100 nnz/row",
    4: "config4: A^2, synthetic cage15-shaped 19-point stencil 172x173x173 (n=5,147,788)",
    5: "config5: conversion + A^2, synthetic R-MAT (see synth.config(5))",
}

# --dump-outputs writes at most this many entries of C (three float64 arrays: 48 MiB)
DUMP_ENTRIES = 1 << 21


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def algorithmic_bytes(a_rows, a_nnz, b_rows, b_nnz, c_rows, c_nnz):
    """SURVEY.md section 8(d): CSR-equivalent compulsory traffic, int32 indices + fp64 values."""
    return 12 * a_nnz + 4 * (a_rows + 1) + 12 * b_nnz + 4 * (b_rows + 1) + 12 * c_nnz + 4 * (c_rows + 1)


class ClockSampler:
    """SM clock and throttle reasons sampled WHILE the timed region runs: NVML from a thread of this
    process (cheap: no extra process hammering the driver), nvidia-smi -lms as the fallback."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    BITS = {"sw_power_cap": 0x4, "hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

    def __init__(self, device):
        self.device, self.rows, self.proc, self.nvml, self.stop_flag = device, [], None, None, False

    def _nvml_handle(self):
        import pynvml
        pynvml.nvmlInit()
        try:
            import torch
            uuid = str(torch.cuda.get_device_properties(self.device).uuid)
            return pynvml, pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
        except Exception:
            return pynvml, pynvml.nvmlDeviceGetHandleByIndex(self.device)

    def start(self):
        try:
            self.nvml, self.handle = self._nvml_handle()
            self.mx = float(self.nvml.nvmlDeviceGetMaxClockInfo(self.handle, self.nvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _poll(self):
        n = self.nvml
        while not self.stop_flag:
            try:
                sm = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
                try:
                    why = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
                except Exception:
                    why = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
                self.rows.append([str(sm), str(self.mx)] + ["Active" if why & bit else "Not Active"
                                                            for bit in (0x8, 0x40, 0x20, 0x4)])
            except Exception:
                pass
            time.sleep(0.02)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.nvml:
            self.stop_flag = True
            self.thread.join(timeout=1)
        elif self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        else:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no NVML and no nvidia-smi"]}
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons), "source": "nvml" if self.nvml else "nvidia-smi"}


def load_workload(k):
    from pem_spgemm_b200 import synth
    name, tb, (rows, cols, I, J, V) = synth.config(k)
    return name, tb, rows, cols, np.ascontiguousarray(I), np.ascontiguousarray(J), np.ascontiguousarray(V)


def oracle_cpu(rows, cols, I, J, V, tb):
    """The host oracle timed on this box's cores (reported baseline, not the target).  All host cores are
    asked for explicitly: torchrun exports OMP_NUM_THREADS=1 to its workers."""
    from oracle import host   # cpu_baseline leg: one of the places allowed to run oracle/
    host.set_threads(os.cpu_count() or 1)
    A = host.coo_to_csr(rows, cols, I, J, V)
    B = host.transpose(A) if tb else A
    flop = host.flop(A, B)
    tm = {}
    host.spgemm(A, B, tm)                      # first run: thread start-up, page faults of the workspaces
    secs, spent = [tm["seconds"]], tm["seconds"]
    while len(secs) < 4 and spent < 20.0:      # up to three more, inside ~20 s of CPU work
        host.spgemm(A, B, tm)
        secs.append(tm["seconds"]); spent += tm["seconds"]
    timed = secs[1:] or secs                   # a run that alone exceeds the budget is its own sample
    return flop, float(np.mean(timed)), tm["threads"], len(timed)


def static_config(k, tb):
    """The `config` object both arms print (same keys, same values: the driver compares them)."""
    return {"workload": CONFIG_TEXT[k], "product": "A*A^T" if tb else "A^2"}


def run_reference(args, rank):
    """--impl reference: the UNMODIFIED reference source (/root/reference/spgemm.cu compiled against shim
    headers, oracle/Makefile) through its own CLI on one B200.  oracle/_ref/pemspgemm_ref61 is built with the
    reference's own virtual architecture (compute_61 PTX, /root/reference/Makefile:13), the only rebuild whose
    NSPARSE step 1 terminates on sm_100 (profiles/r02_reference_runs.md); pemspgemm_ref (compute_100 PTX) is
    tried for inputs that stay on the SPA path.  If no binary is present or both fail on this input (config 2:
    the reference aborts inside thrust; config 5: int32 sizes), the host oracle port on all host cores."""
    if rank != 0:
        return
    import pem_spgemm_b200 as pem
    name, tb, rows, cols, I, J, V = load_workload(args.config)
    line = {"impl": "reference", "metric": "spgemm_gflops", "unit": "GFLOP/s", "n_gpus": 1, "steps": args.steps,
            "warmup": args.warmup, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": static_config(args.config, tb)}
    b_tile_cols = ((rows if tb else cols) + 15) // 16
    nsparse = b_tile_cols > 512 * 32           # /root/reference/spgemm.cu:1142
    bins = ["pemspgemm_ref61"] + ([] if nsparse else ["pemspgemm_ref"])
    failures, done = [], False
    work = f"/tmp/pem_ref_{os.getpid()}"                     # the reference writes its CSV into the working directory
    mtx_dir = "/tmp/pem_ref_mtx"                             # the input file is shared by later invocations on this box
    mtx = os.path.join(mtx_dir, f"{name}.mtx")
    for b in bins:
        ref = os.path.join(ROOT, "oracle", "_ref", b)
        if not os.path.exists(ref):
            failures.append(f"{b}: not built")
            continue
        if args.config == 5:
            failures.append(f"{b}: not launched, nnz(C) = 2.5e9 exceeds the reference's int32 sizes (spgemm.cu:727-728)")
            continue
        os.makedirs(work, exist_ok=True)
        if not os.path.exists(mtx):
            os.makedirs(mtx_dir, exist_ok=True)
            part = f"{mtx}.{os.getpid()}.part"
            pem.mtx_write(part, rows, cols, I, J, V)
            os.replace(part, mtx)
        csv = os.path.join(work, "pemspgemm_benchmark_result.csv")
        if os.path.exists(csv):
            os.remove(csv)
        try:
            t0 = time.time()
            out = subprocess.run([ref, mtx, "0"] + (["1"] if tb else []), cwd=work, capture_output=True, text=True, timeout=420)
            wall = time.time() - t0
            if out.returncode != 0:
                failures.append(f"{b}: rc={out.returncode} {out.stderr.strip()[-200:]}")
                continue
            row = open(csv).read().strip().splitlines()[-1].split(",")
            flop, c_nnz, t_ms, gf = int(row[1]), int(row[2]), float(row[10]), float(row[13])
            if not (t_ms > 0 and c_nnz > 0):
                failures.append(f"{b}: time_ms={t_ms} C_nnz={c_nnz}")
                continue
            line.update({"value": gf, "ms_per_step": t_ms, "steps": 10, "warmup": 1,
                         "reference_binary": b,
                         "reference_csv": {"flop": flop, "C_nnz": c_nnz, "step1_ms": float(row[7]),
                                           "step2_ms": float(row[8]), "step3_ms": float(row[9]),
                                           "kernel_ms": float(row[11]), "malloc_ms": float(row[12])},
                         "cpu_baseline": {"value": gf, "unit": "GFLOP/s", "cores": 0, "kind": "reference",
                                          "sample": f"reference CUDA source rebuilt for sm_100 ({b}), its own CLI: "
                                                    "1 warm-up + 10 timed iterations of the full workload on 1 B200 (it has no CPU path); "
                                                    f"whole process {wall:.1f}s"},
                         "e2e": {"value": gf, "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
            done = True
            break
        except Exception as e:  # timeout, no CSV
            failures.append(f"{b}: {type(e).__name__}: {e}"[:300])
    if failures:
        line["reference_failure"] = "; ".join(failures)
    if not done:
        flop, secs, thr, runs = oracle_cpu(rows, cols, I, J, V, tb)
        gf = 2.0 * flop / secs / 1e9
        line.update({"value": gf, "ms_per_step": secs * 1e3, "steps": runs, "warmup": 1 if runs > 1 or secs < 20 else 0,
                     "cpu_baseline": {"value": gf, "unit": "GFLOP/s", "cores": thr, "kind": "port",
                                      "sample": f"full workload, mean of {runs} run(s) of the OpenMP Gustavson oracle after one warm-up run"},
                     "e2e": {"value": gf, "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
    shutil.rmtree(work, ignore_errors=True)
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", type=int, default=4)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-coo-e2e", action="store_true", help="skip the second end-to-end figure (C pulled to host as sorted COO)")
    ap.add_argument("--keep-empty", type=int, default=0)
    ap.add_argument("--subpanels", type=int, default=0,
                    help="sequential tile-row panels per rank (0 = auto: config 5's C does not fit one GPU in tiled form "
                         "unless it is produced and consumed panel by panel)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write C of the last timed step to DIR/C_{rows,cols,vals}.npy (float64; every entry, or a seeded sample of "
                         f"{DUMP_ENTRIES} positions of the (row, col)-sorted COO when C is larger) and DIR/C_nnz.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    import pem_spgemm_b200 as pem
    from pem_spgemm_b200 import dist as pdist

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    name, tb, rows, cols, I, J, V = load_workload(args.config)
    ctx = pem.Context(local_rank)
    ctx.set_option(pem.OPT_KEEP_EMPTY_TILES, args.keep_empty)
    stream = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", local_rank))

    # operands resident in HBM before the timed region
    tI = torch.from_numpy(I).pin_memory(); tJ = torch.from_numpy(J).pin_memory(); tV = torch.from_numpy(V).pin_memory()
    A = ctx.convert_coo(rows, cols, tI.numpy(), tJ.numpy(), tV.numpy())
    B = ctx.transpose(A) if tb else A
    flop = ctx.count_flop(A, B)
    sub = args.subpanels or (max(1, -(-16 // world)) if args.config == 5 else 1)   # 16 panels: 32-bit sort keys, 416 ms against 658 ms with 8
    bounds = ctx.partition_panels(A, B, world * sub)
    panels = [(int(bounds[rank * sub + i]), int(bounds[rank * sub + i + 1])) for i in range(sub)]

    def barrier():
        ctx.sync()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    tile_products = 0

    def one_step(times=None, kern=None, on_result=None):
        nonlocal tile_products
        nnz = tiles = pairs = tile_products = 0
        for pn in panels:               # this rank's panels, one after the other (results freed in between)
            tp = pem.Times()
            C = ctx.spgemm(A, B, times=tp, panel=pn)
            info = C.info
            nnz += info.nnz; tiles += info.tiles; pairs += info.pairs; tile_products += info.tile_products
            if on_result is not None:
                on_result(C)
            C.free()
            if times is not None:
                for f in ("step1_ms", "step2_ms", "step3_ms"):
                    setattr(times, f, getattr(times, f) + getattr(tp, f))
            if kern is not None:
                for k, v in ctx.kernel_ms().items():
                    kern[k] = kern.get(k, 0.0) + v
        # the path's only exchange: per-shard sizes -> global offsets of every shard of C
        return pdist.exchange_shard_sizes(nnz, tiles, pairs, device="cuda")

    for _ in range(args.warmup):
        layout = one_step()

    # --dump-outputs: positions in the (row, col)-sorted COO of the whole C, seeded, sized from the warm-up's C;
    # this rank takes those inside its own shard from each of its panels during the last timed step
    dump_parts, dump_pauses, dump_launches, seen = [], [], 0, 0
    if args.dump_outputs:
        total = int(layout.totals[0])
        pos = np.arange(total) if total <= DUMP_ENTRIES else np.unique(np.random.default_rng(0).integers(0, total, DUMP_ENTRIES))
        pos = pos[(pos >= layout.nnz_offset) & (pos < layout.nnz_offset + int(layout.sizes[rank, 0]))] - layout.nnz_offset

    def take_sample(C):
        """Copies the sampled entries of one panel's C to the host; the events around the copy take its time out of the step."""
        nonlocal seen, dump_launches
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record(stream)
        n, launched = C.info.nnz, ctx.launch_count
        sel = pos[(pos >= seen) & (pos < seen + n)] - seen
        if sel.size:
            r, c, v = C.to_coo()
            dump_parts.append((r[sel], c[sel], v[sel]))
            del r, c, v                 # unmapping GBs of host memory takes time as well: before the closing event
        seen += n
        dump_launches += ctx.launch_count - launched
        p1.record(stream)
        dump_pauses.append((p0, p1))

    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = ctx.launch_count
    stalls0 = ctx.size_stalls
    step_ms, own_ms, s1, s2, s3, kms = [], [], [], [], [], []
    for step in range(args.steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t = pem.Times()
        e0.record(stream)
        kd = {}
        layout = one_step(t, kd, take_sample if args.dump_outputs and step == args.steps - 1 else None)
        e1.record(stream)
        barrier()
        own = e0.elapsed_time(e1) - sum(p0.elapsed_time(p1) for p0, p1 in dump_pauses)
        ms = torch.tensor([own], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        step_ms.append(float(ms.item()))
        own_ms.append(own)
        s1.append(t.step1_ms); s2.append(t.step2_ms); s3.append(t.step3_ms)
        kms.append(kd)
    launches = ctx.launch_count - launches0 - dump_launches
    stalls = ctx.size_stalls - stalls0
    clocks = sampler.stop() if rank == 0 else None
    c_nnz, c_tiles, c_pairs = (int(x) for x in layout.totals.tolist())
    if args.dump_outputs:
        part = tuple(np.concatenate([p[i] for p in dump_parts]) if dump_parts else np.zeros(0) for i in range(3))
        parts = [part]
        if world > 1:
            parts = [None] * world
            dist.all_gather_object(parts, part)
        if rank == 0:
            os.makedirs(args.dump_outputs, exist_ok=True)
            out = {"C_nnz": np.array([c_nnz])}
            out.update({k: np.concatenate([p[i] for p in parts]) for i, k in enumerate(("C_rows", "C_cols", "C_vals"))})
            for k, a in out.items():
                np.save(os.path.join(args.dump_outputs, k + ".npy"), a.astype(np.float64))
    ms_per_step = float(np.mean(step_ms))
    value = 2.0 * flop / (ms_per_step * 1e6)
    # per-rank figures (imbalance is visible in rank_ms; the dominant kernel's time is the slowest rank's)
    kern_own = {k: float(np.mean([d[k] for d in kms])) for k in kms[0]}
    per_rank = torch.tensor([float(np.mean(own_ms)), float(np.mean(s1)), float(np.mean(s2)), float(np.mean(s3))] +
                            [kern_own[k] for k in sorted(kern_own)] + [float(tile_products)], dtype=torch.float64, device="cuda")
    if world > 1:
        gathered = [torch.zeros_like(per_rank) for _ in range(world)]
        dist.all_gather(gathered, per_rank)
        per_rank_all = torch.stack(gathered).cpu().numpy()
    else:
        per_rank_all = per_rank.cpu().numpy()[None, :]

    # ---- end to end through the C ABI with HOST buffers: H2D of the COO, conversion, SpGEMM, and
    #      (a) D2H of the result summary (sizes + device-reduced checksum) or (b) D2H of C itself as sorted COO
    #      into pinned host buffers (pem_result_to_coo), every step
    e2e_warm = 2            # untimed: the first end-to-end passes grow the memory pool (cudaMalloc inside), like the W warm-up steps
    h2d_rank = 0

    # the host COO stays alive and unmodified for the whole run, so conversion may return while the values are
    # still uploading (PEM_OPT_ASYNC_VALUES): steps 1 and 2 of the product run underneath the upload
    ctx.set_option(pem.OPT_ASYNC_VALUES, 1)

    def e2e_pass(coo_bufs=None):
        nonlocal h2d_rank
        barrier()
        t0 = time.perf_counter()
        if world > 1:       # each rank uploads 1/world of the COO, NVLink all-gather, conversion from device arrays
            dI, dJ, dV, h2d_rank = pdist.upload_coo_sharded(tI, tJ, tV, torch.device("cuda", local_rank))
            torch.cuda.current_stream().synchronize()
            A2 = ctx.convert_coo(rows, cols, dI.data_ptr(), dJ.data_ptr(), dV.data_ptr(), nnz=I.size)
        else:
            A2 = ctx.convert_coo(rows, cols, tI.numpy(), tJ.numpy(), tV.numpy())
        B2 = ctx.transpose(A2) if tb else A2            # A^T from A's tiles, on the device
        pulled = 0
        for pn in panels:
            C2 = ctx.spgemm(A2, B2, panel=pn)
            if coo_bufs is None:
                C2.checksum()
            else:
                n = C2.info.nnz
                assert n <= coo_bufs[0].numel(), "pinned COO buffers too small for this panel"
                C2.to_coo_into(coo_bufs[0].data_ptr(), coo_bufs[1].data_ptr(), coo_bufs[2].data_ptr())
                pulled += 16 * n
            C2.free()
        ctx.sync()
        ms = torch.tensor([(time.perf_counter() - t0) * 1e3, float(pulled)], dtype=torch.float64, device="cuda")
        if world > 1:
            ms_max = ms.clone(); dist.all_reduce(ms_max, op=dist.ReduceOp.MAX)
            dist.all_reduce(ms, op=dist.ReduceOp.SUM)
            ms[0] = ms_max[0]
        if B2 is not A2:
            B2.free()
        A2.free()
        return float(ms[0].item()), int(ms[1].item())

    e2e_ms = [e2e_pass()[0] for _ in range(e2e_warm + args.steps)]
    e2e_t = float(np.mean(e2e_ms[e2e_warm:]))
    h2d = int(I.nbytes + J.nbytes + V.nbytes) if world == 1 else int(h2d_rank) * world
    d2h = (2 * 1024 * 2 * 8 + 3 * 8 * 16) * sub * world    # checksum partials + the size read-backs of one step, all ranks
    e2e_coo = None
    if not args.no_coo_e2e:
        # largest panel of this rank decides the pinned buffer size (panels are flop-balanced: 1.25x the mean is a safe bound, checked)
        cap = int(1.25 * c_nnz / (world * sub)) + (1 << 20)
        bufs = (torch.empty(cap, dtype=torch.int32, pin_memory=True), torch.empty(cap, dtype=torch.int32, pin_memory=True),
                torch.empty(cap, dtype=torch.float64, pin_memory=True))
        runs = [e2e_pass(bufs) for _ in range(1 + args.steps)]
        coo_t = float(np.mean([r[0] for r in runs[1:]]))
        e2e_coo = {"value": 2.0 * flop / (coo_t * 1e6), "unit": "GFLOP/s", "ms_per_step": coo_t,
                   "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": runs[-1][1], "steps": args.steps, "warmup": 1,
                   "what": "as e2e, but C itself is pulled into pinned host buffers as (row, col)-sorted COO through "
                           "pem_result_to_coo: 16 bytes per nonzero of C"}
        del bufs

    if rank == 0:
        peak, peak_src = hbm_peak()
        ai = A.info; bi = B.info
        bytes_alg = algorithmic_bytes(ai.rows, ai.nnz, bi.rows, bi.nnz, ai.rows, c_nnz)
        names = sorted(kern_own)
        rank_ms = [float(x) for x in per_rank_all[:, 0]]
        slow = int(np.argmax(per_rank_all[:, 0]))          # the rank that sets the step time
        t3 = float(per_rank_all[slow, 3])
        step_t = {"step1": float(per_rank_all[slow, 1]), "step2": float(per_rank_all[slow, 2]), "step3": t3}
        # the dominant KERNEL: four kernels are bracketed by CUDA events on the engine's own stream inside
        # pem_spgemm (pem_ctx_kernel_ms); their averages over the timed steps are taken live, here (slowest rank)
        kern_t = {k: float(per_rank_all[slow, 4 + i]) for i, k in enumerate(names)}
        dom = max(kern_t, key=kern_t.get)
        sort_passes = ctx.last_sort_passes
        dom_kernel = {"k_expand": "k_expand (step 1: tile-product expansion + occupancy filter)",
                      "radix_sort": ("no sort (per-row bitmap path of step 1)" if sort_passes < 0 else
                                     "k_row_sort (step 1: block-local bitonic sort of each C' row's tile pairs)" if sort_passes == 0 else
                                     f"cub::DeviceRadixSort onesweep, {sort_passes} passes (step 1: sort of the kept tile pairs)"),
                      "k_step2_pairs": "k_step2_pairs (step 2: 16x16 boolean products, pair-parallel)",
                      "step3_numeric": {4: "k_step3_windows (step 3: fp64 numeric accumulation, pair records staged in shared memory)",
                                        3: "k_step3_classes (step 3: fp64 numeric accumulation, tile classes)",
                                        1: "k_step3_numeric (step 3: fp64 numeric accumulation, row-owner)"}.get(
                                            ctx.last_step3_kernel, "k_step3_entries (step 3: fp64 numeric accumulation)")}[dom]
        td = kern_t[dom]
        # compulsory bytes of each timed kernel (DESIGN.md section 3), whole job; the numeric kernel's are the
        # algorithmic bytes of the product (SURVEY.md 8d: it reads A and B and writes C)
        P = int(per_rank_all[:, -1].sum())
        kernel_bytes = {"k_expand": 2 * P + 12 * c_pairs,
                        "radix_sort": 2 * 12 * c_pairs * max(1, sort_passes),
                        "k_step2_pairs": (8 + 64 + 4) * c_pairs + 32 * c_tiles,
                        "step3_numeric": bytes_alg}
        kb = kernel_bytes[dom]
        traffic = None
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json"))).get(f"config{args.config}", {}).get(dom)
        except Exception:
            pass
        line = {
            "metric": "spgemm_gflops", "value": value, "unit": "GFLOP/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": static_config(args.config, tb),
            "workload_stats": {"flop": flop, "nnz_A": int(ai.nnz), "nnz_C": c_nnz, "C_tiles": c_tiles, "tile_pairs": c_pairs,
                               "parallelism": f"tile-row panels x{world}, B replicated" + (f"; {sub} sequential sub-panels per GPU" if sub > 1 else ""),
                               "l2": "no flush: each step streams > 1 GB (C + C' metadata), far above the 126 MB L2",
                               "keep_empty_tiles": args.keep_empty},
            "rank_ms": rank_ms,
            "step_ms": step_t, "kernel_ms": kern_t,
            # at N GPUs the job's bytes are split over N kernels running side by side: the peak is N x one GPU's
            "roofline": {"bound": "hbm", "kernel": dom_kernel, "achieved": kb / (td * 1e6) if td > 0 else None,
                         "peak": peak * world, "unit": "GB/s", "frac": (kb / (td * 1e6) / (peak * world)) if td > 0 else None,
                         "traffic": traffic, "algorithmic_bytes": bytes_alg, "kernel_bytes": kb, "peak_source": peak_src + (f" x {world} GPUs" if world > 1 else ""),
                         "numeric_kernel_frac": (bytes_alg / (kern_t["step3_numeric"] * 1e6) / (peak * world)) if kern_t.get("step3_numeric", 0) > 0 else None,
                         "whole_spgemm_frac": bytes_alg / (ms_per_step * 1e6) / (peak * world)},
            "e2e": {"value": 2.0 * flop / (e2e_t * 1e6), "unit": "GFLOP/s", "ms_per_step": e2e_t,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": len(e2e_ms) - e2e_warm, "warmup": e2e_warm,
                    "what": "host COO (pinned) -> pem_convert_coo (values upload overlapped with the symbolic steps) -> pem_spgemm -> checksum/sizes read back"
                            + ("; every rank uploads 1/N of the COO and the slices are all-gathered over NVLink" if world > 1 else "")},
            "gpu_launches": int(launches),
            "host_stalls_in_timed_steps": int(stalls),     # size read-backs that stalled the host (0: the warm-up steps recorded the size plans)
            "clocks": clocks,
        }
        if e2e_coo is not None:
            line["e2e_coo"] = e2e_coo
        if world == 1 and not args.no_cpu_baseline:
            f2, secs, thr, runs = oracle_cpu(rows, cols, I, J, V, tb)
            assert f2 == flop, "engine and oracle disagree on flop"
            line["cpu_baseline"] = {"value": 2.0 * flop / secs / 1e9, "unit": "GFLOP/s", "cores": thr, "kind": "port",
                                    "sample": f"full workload, mean of {runs} run(s) of the OpenMP Gustavson oracle (symbolic + numeric) after one warm-up run"}
        print(json.dumps(line), flush=True)
    if B is not A:
        B.free()
    A.free()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
