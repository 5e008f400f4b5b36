#!/usr/bin/env python
"""bench.py — benchmark of the hot path (BASELINE.json): rows/s of cudf::sort_by_key on a 1e9-row int64 column
(configs[1]) per GPU through the pylibcudf-named shim over the C ABI, plus (N = 1) the other operations BASELINE's metric
names — hash inner_join (configs[2]), groupby (configs[3]), scan / reduce — as sub-objects under `ops`, and (N > 1) the
sharded inner_join (configs[4]) under `sharded_inner_join`.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--rows R] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one sort_by_key(values=T, keys=T) over a resident synthetic column (splitmix64 keys, SURVEY §8d); at N > 1
the sharded sort (sample -> splitters -> range partition -> bucket exchange over NVLink -> local sort).
`value` is device-resident throughput.  `e2e` is the same call fed from PINNED HOST memory with the sorted column copied
back to pinned host memory, every step, inside the timed region; the steps are software-pipelined over three streams
(H2D of step i+1 and D2H of step i-1 overlap the sort of step i; PCIe is full duplex).
`roofline` is measured live with CUDA events around the one-sweep pass launches (b2_profile_*).
`cpu_baseline` / `--impl reference` time pandas (configs[0], the reference's CPU-runnable case) on a bounded 1e7-row
sample of the same key stream on the host cores.
Inputs (8 GB per GPU) are far larger than the 126 MB L2, so no explicit L2 flush is needed.
`--dump-outputs DIR` writes the sorted column of the last timed step as DIR/sorted_keys.npy (float64; at N > 1 one file per
rank, sorted_keys_rank<r>.npy): every row when the output fits DUMP_BYTES, else the rows at a fixed, seeded set of positions
(ascending; see dump_sorted). The inputs depend only on the arguments, so two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True  # the benchmark leaves the tree as it found it (which may be read-only)

METRIC = "sort_by_key_rows_per_s"
UNIT = "rows/s"
SEED_KEYS = 0x5EED0001  # SURVEY §8d seed of the key stream (same constant as oracle/datagen.py; the GPU arm does not import oracle)
DUMP_BYTES = 32 << 20  # --dump-outputs: float64 values per run, summed over ranks
DUMP_SEED = 0x5EED00D0


def _positive(s: str) -> int:
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError("must be at least 1")
    return v


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=_positive, default=5, help="timed steps")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rows", type=int, default=1_000_000_000, help="rows per GPU")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-rows", type=int, default=10_000_000)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-ops", action="store_true", help="skip the per-operation measurements (join / groupby / scan / reduce) at N = 1")
    ap.add_argument("--no-join", action="store_true", help="skip the sharded inner_join measurement at N > 1")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the sorted column of the last timed step under DIR (.npy)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs; the reference arm times a CPU sample")
    return args


# ------------------------------------------------------------------------------------------------
# CPU baseline (pandas; the oracle's host-side twin of the workload) — the one leg that may import oracle/
# ------------------------------------------------------------------------------------------------
def cpu_sort_sample(cpu_rows: int, steps: int, warmup: int):
    import numpy as np
    import pandas as pd

    from oracle import datagen

    keys = datagen.fill(cpu_rows, datagen.SEED_KEYS, 0, 0)
    df = pd.DataFrame({"k": keys})
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        out = df.sort_values("k", kind="stable")
        t1 = time.perf_counter()
        if i >= warmup:
            times.append(t1 - t0)
    assert bool(np.all(np.diff(out["k"].to_numpy()) >= 0))
    best = min(times)
    # other host implementations of the same sort on the same sample (one run each; reported, not the baseline value)
    alt = {}
    try:
        t0 = time.perf_counter()
        np.sort(keys, kind="stable")
        alt["numpy_stable_sort_rows_per_s"] = cpu_rows / (time.perf_counter() - t0)
        import pyarrow as pa
        import pyarrow.compute as pc

        arr = pa.array(keys)
        t0 = time.perf_counter()
        pc.take(arr, pc.sort_indices(arr))
        alt["pyarrow_sort_indices_take_rows_per_s"] = cpu_rows / (time.perf_counter() - t0)
        alt["pyarrow_threads"] = pa.cpu_count()
    except Exception as ex:  # optional extras only
        alt["error"] = repr(ex)[:120]
    return {
        "value": cpu_rows / best,
        "unit": UNIT,
        "cores": 1,  # pandas/numpy sort is single-threaded
        "kind": "port",
        "sample": f"pandas {pd.__version__} DataFrame.sort_values(kind='stable') on {cpu_rows} int64 rows "
                  f"(same splitmix64 key stream), best of {steps}; host has {os.cpu_count()} logical cores",
        "ms": best * 1e3,
        "alternatives": alt,
    }, sum(times) / len(times)


def workload_config(n: int, world: int) -> dict:
    return {"workload": f"{n}-row single int64 column sort_by_key(values=T, keys=T), no nulls, ASCENDING, per GPU "
                        "(BASELINE.json configs[1])" + ("" if world == 1 else f"; sharded over {world} GPUs: sample-sort splitters, stable range "
                        "partition, bucket exchange over NVLink peer memory (fused scatter at 2 ranks, partition + contiguous peer "
                        "copies above), local radix sort (configs[4])"),
            "rows_per_gpu": n, "l2_flush": "inputs (8 GB/GPU) exceed the 126 MB L2; no explicit flush",
            "generator": "splitmix64(seed 0x5EED0001 + i)"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = max(1, args.steps), max(0, min(args.warmup, 2))
    base, mean_s = cpu_sort_sample(args.cpu_rows, steps, warmup)
    line = {
        "impl": "reference",
        "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
        "ms_per_step": mean_s * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int64", "data": "synthetic",
        "config": dict(workload_config(args.rows, max(1, args.gpus)),
                       sample=f"each step = pandas DataFrame.sort_values(kind='stable') on a {args.cpu_rows}-row sample of the key "
                              "stream (BASELINE.json configs[0]: the reference's CPU-runnable case)", rows_per_step=args.cpu_rows),
        "cpu_baseline": base,
        "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# clocks sampler
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.samples = []
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        try:
            p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                  "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            return
        try:
            while not self._stop.is_set():
                line = p.stdout.readline()
                if not line:
                    break
                self.samples.append([x.strip() for x in line.split(",")])
        finally:
            p.terminate()

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._t:
            self._t.join(timeout=2)

    def summary(self):
        sm, mx, reasons = [], [], set()
        for s in self.samples:
            try:
                sm.append(float(s[1]))
                mx.append(float(s[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm_sorted = sorted(sm)
        # "under load": upper half of the samples (the sampler also sees the idle gaps between steps)
        load = sm_sorted[len(sm_sorted) // 2:]
        return {"sm_mhz": load[len(load) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def measured_traffic(kernel_key: str):
    """DRAM bytes per row of one launch of the dominant kernel, from this round's `ncu --set full` capture
    (profiles/r2_traffic.json: dram__bytes_read.sum + dram__bytes_write.sum at 2^27 rows)."""
    p = ROOT / "profiles" / "r2_traffic.json"
    try:
        e = json.loads(p.read_text())[kernel_key]
        return float(e["dram_bytes_per_row"]), (f"profiles/r2_traffic.json[{kernel_key}] ({e.get('source', 'ncu --set full')}), "
                                                "per-row figure x rows of one launch")
    except Exception:
        return None, "no ncu capture of this kernel under profiles/ yet"


def dump_sorted(out_dir: str, col, rank: int, world: int) -> None:
    """Writes `col` (the int64 CUDA tensor a caller of the timed step receives) as float64 .npy under out_dir: all of it up to
    cap = DUMP_BYTES // world // 8 rows, else its values at the ascending positions
    np.unique(default_rng(DUMP_SEED + rank).integers(0, len(col), cap)), which depend only on the row count."""
    import numpy as np
    import torch

    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    n, cap = col.numel(), DUMP_BYTES // world // 8
    if n > cap:
        rows = np.unique(np.random.default_rng(DUMP_SEED + rank).integers(0, n, cap))
        col = col[torch.from_numpy(rows).to(col.device)]
    name = "sorted_keys.npy" if world == 1 else f"sorted_keys_rank{rank}.npy"
    np.save(d / name, col.cpu().numpy().astype(np.float64))


def pin_to_gpu_numa_node(gpu_index: int):
    """Bind this process to the CPUs of the NUMA node its GPU hangs off, before the pinned host buffers are allocated (they are then
    placed on that node): the e2e copies of 8 ranks otherwise cross the host's socket interconnect. Returns a short note."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(gpu_index)], capture_output=True, text=True,
                             timeout=20).stdout.strip()
        bdf = out.lower()
        if bdf.count(":") == 2 and len(bdf.split(":")[0]) == 8:   # 00000000:1B:00.0 -> 0000:1b:00.0
            bdf = bdf[4:]
        node = int(Path(f"/sys/bus/pci/devices/{bdf}/numa_node").read_text().strip())
        if node < 0:
            return "numa: single node"
        cpus = set()
        for part in Path(f"/sys/devices/system/node/node{node}/cpulist").read_text().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if allowed:
            os.sched_setaffinity(0, allowed)
            return f"numa: node {node}, {len(allowed)} cpus"
        return "numa: no allowed cpu on the GPU's node"
    except Exception as ex:  # best effort
        return f"numa: not pinned ({type(ex).__name__})"


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def run_ours(args):
    import ctypes as C

    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    numa_note = pin_to_gpu_numa_node(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    import __graft_entry__ as g

    g.build()
    import cudf_b200.pylibcudf as plc
    from cudf_b200 import _lib

    n = args.rows
    dev = torch.device("cuda", local_rank)
    stream = torch.cuda.current_stream()
    keys = torch.empty(n, dtype=torch.int64, device=dev)
    # disjoint counter range per rank: rank r draws x_i for i in [r*n, (r+1)*n)
    _lib.check(_lib.lib.b2_fill_splitmix64(C.c_void_p(keys.data_ptr()), n, SEED_KEYS, rank * n, 0, 0, _lib.stream_arg(None)))
    torch.cuda.synchronize()

    sharded = None
    if world > 1:
        from cudf_b200 import sharded

        def step():
            return sharded.sort_by_key_sharded(keys, keys)
    else:
        col = plc.Column.from_torch(keys)
        tbl = plc.Table([col])

        def step():
            return plc.sorting.sort_by_key(tbl, tbl, [plc.Order.ASCENDING], [])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for _ in range(max(args.warmup, 3)):
        out = step()
        del out
    barrier()

    # ---- timed region: device-resident ----
    _lib.lib.b2_profile_reset()
    _lib.lib.b2_profile_enable(1)
    launches0 = _lib.kernel_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clocks:
        barrier()
        e0.record(stream)
        for _ in range(args.steps):
            out = None  # the previous step's output is released before this step allocates its own
            out = step()
        e1.record(stream)
        barrier()
    _lib.lib.b2_profile_enable(0)
    if args.dump_outputs:
        dump_sorted(args.dump_outputs, out if world > 1 else out.columns()[0].to_torch(), rank, world)
    del out
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    launches = _lib.kernel_launch_count() - launches0
    ms_step = ms_total / args.steps
    value = world * n / (ms_step / 1e3)

    # ---- live roofline of the dominant kernel (one-sweep pass) ----
    peaks_path = ROOT / "MEASURED_PEAKS.json"
    peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    if peaks_path.exists():
        try:
            peak = float(json.loads(peaks_path.read_text())["hbm_gbs"])
            peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    os_all_ms, os_all_cnt = _lib.profile_get("onesweep")
    # the host launches one kernel per digit; passes the plan skipped (hybrid plan: the low digits; trivial digits) return at
    # once — only launches of at least 0.2 ms (at >= 1e8 rows) are executed passes
    min_ms = 0.2 if n >= 100_000_000 else 0.0
    os_ms, os_cnt = _lib.profile_get_over("onesweep", min_ms)
    hist_ms, _ = _lib.profile_get("histogram")
    ga_ms, _ = _lib.profile_get("gather")
    fix_ms, fix_cnt = _lib.profile_get_over("segment_fix", min_ms)
    rows_local = n  # per rank; at N > 1 the received shard differs from n by < 1 % (sample-sort splitters)
    carry = os.environ.get("B2_SORT_CARRY", "1") != "0"
    hybrid = fix_cnt > 0
    if carry:
        sort_path, pass_bytes_row, kernel_name, tkey = ("(key, 8-byte payload) carried through the passes", 32.0,
                                                        "onesweep_kernel<uint64,(key,8-byte payload)>", "onesweep_carry")
    else:
        sort_path, pass_bytes_row, kernel_name, tkey = "(key, row id) passes + gather", 24.0, "onesweep_kernel<uint64,(key,row id)>", "onesweep_rowid"
    sort_path += "; hybrid plan: LSD passes over the top digits, then the segment fix-up" if hybrid else "; full LSD"
    roofline = None
    if os_cnt and rows_local:
        passes_per_step = os_cnt / args.steps
        per_launch_bytes = pass_bytes_row * rows_local
        avg_ms = os_ms / os_cnt
        achieved = per_launch_bytes / (avg_ms / 1e3) / 1e9
        tr_row, tr_src = measured_traffic(tkey)
        # algorithmic bytes of THIS implementation per row: histogram 8 + executed passes + fix-up (key + payload in, payload out) / gather
        impl_bytes_row = 8 + passes_per_step * pass_bytes_row + (24 if hybrid and carry else (16 if hybrid else 0)) + (0 if carry else 20)
        roofline = {
            "bound": "hbm", "kernel": kernel_name, "sort_path": sort_path, "achieved": achieved, "peak": peak, "unit": "GB/s",
            "frac": achieved / peak,
            "traffic": tr_row * rows_local if tr_row else None, "traffic_source": tr_src,
            "peak_source": peak_src, "rank": rank,
            "algorithmic_bytes_per_launch": per_launch_bytes, "algorithmic_bytes_per_row_per_launch": pass_bytes_row,
            "avg_launch_ms": avg_ms, "launches": os_cnt, "executed_passes_per_step": passes_per_step,
            "launches_incl_skipped_and_sample_sort": os_all_cnt,
            "kernel_share_of_step": os_ms / ms_total,
            "whole_op": {"algorithmic_bytes_per_row_contract": 216, "achieved_GBps_contract": 216.0 * rows_local / (ms_step / 1e3) / 1e9,
                         "frac_contract": 216.0 * rows_local / (ms_step / 1e3) / 1e9 / peak,
                         "algorithmic_bytes_per_row_this_algorithm": impl_bytes_row,
                         "frac_this_algorithm": impl_bytes_row * rows_local / (ms_step / 1e3) / 1e9 / peak,
                         "note": "contract = SURVEY §8d C2 formula (8-bit LSD, row ids + gather: 216 B/row); this algorithm moves fewer bytes "
                                 "(BASELINE.md §2 restates its formula)"},
            "other_kernels_ms_per_step": {"histogram": hist_ms / args.steps, "gather": ga_ms / args.steps, "segment_fix": fix_ms / args.steps,
                                          "onesweep_total": os_all_ms / args.steps},
        }

    # ---- N > 1: per-phase device times of the sharded step (CUDA events inside sharded.py), max over ranks ----
    phases_ms = None
    if world > 1:
        sharded.enable_phase_timing(True)
        acc = {}
        reps = 3
        for _ in range(reps):
            barrier()
            out = step()
            ph = sharded.phases()
            del out
            for k_, v_ in ph.items():
                acc[k_] = acc.get(k_, 0.0) + v_ / reps
        sharded.enable_phase_timing(False)
        names = sorted(acc)
        vals = torch.tensor([acc[k_] for k_ in names], dtype=torch.float64, device=dev)
        dist.all_reduce(vals, op=dist.ReduceOp.MAX)
        phases_ms = {k_: float(v_) for k_, v_ in zip(names, vals.tolist())}

    # ---- e2e: pinned host -> device -> sort_by_key -> pinned host, software-pipelined over three streams ----
    e2e = None
    if not args.no_e2e:
        try:
            cap = n if world == 1 else int(n * 1.1) + 1024  # a rank's shard of the sharded result is ~n rows
            alloc_err = None
            try:
                h_in = torch.empty(n, dtype=torch.int64, pin_memory=True)
                h_out = [torch.empty(cap, dtype=torch.int64, pin_memory=True) for _ in range(2)]
                d_in = [torch.empty(n, dtype=torch.int64, device=dev) for _ in range(2)]
            except Exception as ex:  # e.g. not enough pinnable host memory on this rank
                alloc_err = ex
            ok = torch.tensor([0 if alloc_err else 1], dtype=torch.int32, device=dev)
            if world > 1:  # every rank must take the same branch, or the collectives below would hang
                dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if int(ok.item()) == 0:
                raise RuntimeError(f"e2e buffers could not be allocated on every rank: {alloc_err!r}")
            h_in.copy_(keys)
            torch.cuda.synchronize()
            s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()

            def pipeline(k):
                """k steps; step i: H2D (copy-in stream) -> sort (compute stream) -> D2H (copy-out stream). Buffers are
                double-buffered; events order the three streams. Every step's copies are issued inside the timed region."""
                in_ready = [None, None]
                in_free = [None, None]
                out_done = [None, None]
                outs = [None, None]
                for i in range(k):
                    b = i & 1
                    with torch.cuda.stream(s_in):
                        if in_free[b] is not None:
                            s_in.wait_event(in_free[b])       # the sort that read this buffer two steps ago has finished
                        d_in[b].copy_(h_in, non_blocking=True)
                        in_ready[b] = torch.cuda.Event()
                        in_ready[b].record(s_in)
                    stream.wait_event(in_ready[b])
                    if out_done[b] is not None:
                        # D2H of step i-2 has finished: pinned buffer b is free, and that step's device output may be released
                        # (its stream-ordered free lands on the compute stream behind this wait)
                        stream.wait_event(out_done[b])
                        outs[b] = None
                    if world == 1:
                        c = plc.Column.from_torch(d_in[b])
                        o = plc.sorting.sort_by_key(plc.Table([c]), plc.Table([c]), [plc.Order.ASCENDING], [])
                        res = o.columns()[0].to_torch()
                    else:
                        o = sharded.sort_by_key_sharded(d_in[b], d_in[b])
                        res = o
                    in_free[b] = torch.cuda.Event()
                    in_free[b].record(stream)
                    with torch.cuda.stream(s_out):
                        s_out.wait_event(in_free[b])
                        m = min(res.numel(), cap)
                        h_out[b][:m].copy_(res[:m], non_blocking=True)
                        out_done[b] = torch.cuda.Event()
                        out_done[b].record(s_out)
                    outs[b] = (o, res)
                for ev in out_done:
                    if ev is not None:
                        stream.wait_event(ev)
                return outs

            keep = pipeline(2)
            torch.cuda.synchronize()
            del keep
            k = max(2, min(args.steps, 16))  # fill (first H2D) and drain (last D2H) of the pipeline stay inside the timed region
            barrier()
            e0.record(stream)
            keep = pipeline(k)
            e1.record(stream)
            barrier()
            ems = max_over_ranks(e0.elapsed_time(e1) / k)
            del keep
            assert bool((h_out[0][1:1000001] >= h_out[0][:1000000]).all()) and bool((h_out[1][1:1000001] >= h_out[1][:1000000]).all())
            e2e = {"value": world * n / (ems / 1e3), "unit": UNIT, "h2d_bytes_per_step": 8 * n * world,
                   "d2h_bytes_per_step": 8 * n * world, "ms_per_step": ems, "steps": k, "host_placement": numa_note,
                   "pipeline": "three streams, double-buffered: H2D(i+1) | sort(i) | D2H(i-1); every step copies its 8 GB/GPU input from "
                               "pinned host memory and its sorted 8 GB/GPU output back to pinned host memory inside the timed region"}
            del h_in, h_out, d_in
        except Exception as ex:  # e.g. not enough pinnable host memory
            e2e = {"value": None, "unit": UNIT, "error": repr(ex)[:200]}

    # ---- N > 1: sharded inner_join (BASELINE configs[4]) ----
    sjoin = None
    if world > 1 and not args.no_join:
        try:
            del keys
            _lib.check(_lib.lib.b2_trim_pool())
            sjoin = bench_sharded_join(args, torch, dist, sharded, _lib, C, n, world, rank, dev, barrier, max_over_ranks)
        except Exception as ex:
            sjoin = {"error": repr(ex)[:300]}

    ops = None
    if world == 1 and not args.no_ops:
        import bench_extra

        del keys, col, tbl
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        _lib.check(_lib.lib.b2_trim_pool())
        try:
            ops = bench_extra.run(plc, _lib, n, peak, cpu_rows=args.cpu_rows)
        except Exception as ex:
            ops = {"error": repr(ex)[:300]}

    if rank == 0:
        cpu_base, _ = cpu_sort_sample(args.cpu_rows, 3, 1)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64",
            "data": "synthetic",
            "config": workload_config(n, world),
            "roofline": roofline, "cpu_baseline": cpu_base, "e2e": e2e, "gpu_launches": int(launches),
            "clocks": clocks.summary(),
        }
        if phases_ms is not None:
            line["phases_ms"] = phases_ms
        if sjoin is not None:
            line["sharded_inner_join"] = sjoin
        if ops is not None:
            line["ops"] = ops
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def bench_sharded_join(args, torch, dist, sharded, _lib, C, n, world, rank, dev, barrier, max_over_ranks):
    """configs[4]: inner_join of two row-sharded int64 key columns, n rows per GPU and side, 10 % of the probe rows match a
    build row (of another rank) exactly once: hash partition of (key, global row id) on both sides -> bucket exchange ->
    local join -> global row-id pairs. Row-id consistency is checked on the result (as scripts/sharded_check.py does)."""
    def fill(t, seed, first):
        _lib.check(_lib.lib.b2_fill_splitmix64(C.c_void_p(t.data_ptr()), t.numel(), seed, first, 0, 0, _lib.stream_arg(None)))
        return t

    m = n
    rk = fill(torch.empty(m, dtype=torch.int64, device=dev), 0x5EED0002, rank * m)
    # probe rank r: every 10th row copies the key of the same row of build rank (r+1) % world; the other rows are fresh keys
    lk = fill(torch.empty(m, dtype=torch.int64, device=dev), 0x5EED0009, (1 << 45) + rank * m)
    nxt = (rank + 1) % world
    chunk = 50_000_000  # multiple of 10: the strided rows line up with the chunk starts
    for c0 in range(0, m, chunk):
        c1 = min(m, c0 + chunk)
        tmp = fill(torch.empty(c1 - c0, dtype=torch.int64, device=dev), 0x5EED0002, nxt * m + c0)
        lk[c0:c1:10] = tmp[::10]
        del tmp
    expected_local = len(range(0, m, 10))

    def step():
        return sharded.inner_join_sharded(lk, rk)

    jl, jr = step()
    torch.cuda.synchronize()
    tot = torch.tensor([jl.numel()], dtype=torch.int64, device=dev)
    dist.all_reduce(tot)
    lrank, lrow = jl // m, jl % m
    consistent = bool((lrow % 10 == 0).all()) and bool((jr == ((lrank + 1) % world) * m + lrow).all())
    okc = torch.tensor([1 if consistent else 0], dtype=torch.int32, device=dev)
    dist.all_reduce(okc, op=dist.ReduceOp.MIN)
    del jl, jr, lrank, lrow
    k = max(1, min(args.steps, 3))
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(k):
        o = step()
        del o
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1) / k)
    sharded.enable_phase_timing(True)
    barrier()
    o = step()
    ph = sharded.phases()
    del o
    sharded.enable_phase_timing(False)
    names = sorted(ph)
    vals = torch.tensor([ph[k_] for k_ in names], dtype=torch.float64, device=dev)
    dist.all_reduce(vals, op=dist.ReduceOp.MAX)
    return {"metric": "sharded_inner_join_probe_rows_per_s", "value": world * m / (ms / 1e3), "unit": "probe rows/s", "ms_per_step": ms, "steps": k,
            "rows_per_gpu_per_side": m, "pairs": int(tot.item()), "pairs_expected": world * expected_local,
            "row_ids_consistent": bool(int(okc.item())), "phases_ms": {k_: float(v_) for k_, v_ in zip(names, vals.tolist())},
            "workload": f"inner_join of two int64 key columns, {m} rows per GPU and side, 10 % of probe rows match once; (key, global row id) "
                        "hash-partitioned and exchanged over NVLink peer memory, local join, global row-id pairs (BASELINE configs[4])"}


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
