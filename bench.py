#!/usr/bin/env python
"""bench.py -- rows/s of the windowed group-aggregate hot path on synthetic sensor batches (BASELINE.json metric).

Own arm   : `python bench.py --gpus N --steps K --warmup W`   (N>1: one rank per GPU under torchrun)
Reference : `python bench.py --impl reference ...`            (the CPU restatement of the reference algorithm -- the Rust
            reference cannot be built in this image -- on all host cores; rank 0 only)

A "step" is one pass of the operator over the whole synthetic stream of the workload (configs[1] of BASELINE.json:
tumbling 1 s, key sensor_name, count/min/max/avg(reading), 1e9 rows, 100K groups, 64Ki-row batches) with a fresh
operator handle: push every batch, close the last window, collect the emitted rows.
  value : inputs already resident in HBM (dnz_window_push_device / poll_device), device timed with CUDA events on the
          stream the kernels run on.
  e2e   : the same metric through the reference-facing C ABI with HOST Arrow buffers in pinned memory
          (dnz_window_push / dnz_window_poll): host->device copies of the inputs and device->host copies of the emitted
          rows are inside the timed region.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

T0 = 1_700_000_000_000
WORKLOADS = {
    # name: (rows, groups, rows_per_ms, window_ms, slide_ms, filter, uuid_keys)
    "cfg1": dict(rows=10_000_000, groups=1_000, rows_per_ms=1_000, window_ms=1000, slide_ms=0, filt=None, uuid=False),
    "cfg2": dict(rows=1_000_000_000, groups=100_000, rows_per_ms=10_000, window_ms=1000, slide_ms=0, filt=None, uuid=False),
    "cfg3": dict(rows=1_000_000_000, groups=1_000_000, rows_per_ms=10_000, window_ms=10_000, slide_ms=1000, filt=None, uuid=False),
    "cfg4": dict(rows=1_000_000_000, groups=100_000, rows_per_ms=10_000, window_ms=1000, slide_ms=0, filt=("max", ">", 113.0), uuid=False),
    # experiment only (not a BASELINE config): cfg2 with ONE pane for the whole stream -- isolates pane-boundary effects
    "cfg2w": dict(rows=1_000_000_000, groups=100_000, rows_per_ms=10_000, window_ms=1_000_000, slide_ms=0, filt=None, uuid=False),
    "cfg5": dict(rows=1_000_000_000, groups=10_000_000, rows_per_ms=8_000, window_ms=60_000, slide_ms=5000, filt=None, uuid=True),
}
BATCH_ROWS = 65536
AGGS = [("count", "reading", "count"), ("min", "reading", "min"), ("max", "reading", "max"), ("avg", "reading", "average")]


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="own", choices=["own", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--rows", type=int, default=0, help="override the workload's row count (debugging only)")
    ap.add_argument("--e2e-rows", type=int, default=0, help="rows of the stream fed from host memory in the e2e leg (0 = auto)")
    ap.add_argument("--cpu-rows", type=int, default=0, help="rows of the CPU-baseline sample (0 = auto, ~10-30 s)")
    ap.add_argument("--max-rows-per-launch", type=int, default=0)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-exchange", action="store_true", help="N>1: skip the extra leg with un-partitioned input + pane all-to-all")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle comparison of the legs' output (outside the timed regions)")
    ap.add_argument("--flags", type=int, default=0, help="extra DNZ_FLAG_* bits for the operator (experiments)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the rows the last of them emitted to DIR/<column>.npy (see dump_outputs)")
    return ap.parse_args()


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "25",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); smax.append(float(r[2]))
                for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU legs (the oracle is the checker / baseline here, never the thing shipped)
def cpu_baseline(wl, rows, threads):
    """Times the multi-threaded CPU restatement of the reference algorithm on a bounded sample of the workload."""
    from oracle import OracleMT, synth_batch
    from tests.helpers import rows_to_batch
    nb = max(1, rows // BATCH_ROWS)
    batches = [synth_batch(i * BATCH_ROWS, BATCH_ROWS, groups=wl["groups"], rows_per_ms=wl["rows_per_ms"], uuid_keys=wl["uuid"],
                           extra_columns=True) for i in range(nb)]
    last = int(batches[-1].ts[-1])
    # closing batch: one row per key would be needed per partition in the reference; the deterministic shared watermark of
    # the restatement lets a single sentinel row close every partition's windows
    batches.append(rows_to_batch([((last // 1000 + 1) * 1000 + 2 * wl["window_ms"], 1.0, b"sentinel")]))
    m = OracleMT(wl["window_ms"], wl["slide_ms"], wl["filt"], partitions=threads)
    t = time.perf_counter()
    m.push_many(batches)
    dt = time.perf_counter() - t
    out_rows = m.num_results()
    m.close()
    return nb * BATCH_ROWS / dt, dt, nb * BATCH_ROWS, out_rows


_best_threads = {}


def choose_threads(wl):
    """The reference would run target_partitions = #cores; the restatement is given whichever partition count in
    {cores, cores/2, cores/4, cores/8} is fastest on a short calibration sample (generous to the CPU side)."""
    cores = os.cpu_count() or 1
    key = (wl["groups"], wl["window_ms"], wl["slide_ms"])
    if key in _best_threads:
        return _best_threads[key]
    cands = sorted({max(1, cores // d) for d in (1, 2, 4, 8)}, reverse=True)
    best, best_rate = cands[0], 0.0
    if len(cands) > 1:
        for t in cands:
            rate, _, _, _ = cpu_baseline(wl, BATCH_ROWS * 96, t)
            if rate > best_rate:
                best, best_rate = t, rate
    _best_threads[key] = best
    return best


def auto_cpu_rows(wl, threads):
    # ~10-30 s of CPU work: single-thread rate of the restatement is ~5-10 M rows/s per overlapping window
    per_row_windows = max(1, wl["window_ms"] // (wl["slide_ms"] or wl["window_ms"]))
    est_rate = 5e6 * min(threads, 64) / per_row_windows
    return int(max(BATCH_ROWS * 8, min(200_000_000, est_rate * 15)) // BATCH_ROWS * BATCH_ROWS)


def run_reference(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = choose_threads(wl)
    rows = args.cpu_rows or auto_cpu_rows(wl, threads)
    rates = []
    for i in range(args.warmup + args.steps):
        rate, dt, n, _ = cpu_baseline(wl, rows, threads)
        if i >= args.warmup:
            rates.append((rate, dt))
    value = float(np.mean([r for r, _ in rates]))
    sample = f"{rows} rows ({rows // BATCH_ROWS} batches of {BATCH_ROWS}) of the {args.workload} stream per step"
    line = {"impl": "reference", "metric": "rows/sec windowed group-agg on synthetic sensor batches", "value": value, "unit": "rows/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": float(np.mean([d for _, d in rates]) * 1e3),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args, wl, 1),
            "cpu_baseline": {"value": value, "unit": "rows/s", "cores": threads, "threads": threads, "host_cores": os.cpu_count(), "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "CPU restatement of the reference algorithm (oracle/, hash-partitioned over all host cores); the Rust "
                    "reference itself cannot be built in this image"}
    print(json.dumps(line), file=claim_stdout(), flush=True)


def workload_config(args, wl, world):
    return {"workload": f"{args.workload}: {'tumbling' if not wl['slide_ms'] else 'sliding'} {wl['window_ms']}ms"
                        f"{'/' + str(wl['slide_ms']) + 'ms' if wl['slide_ms'] else ''}, key sensor_name, count/min/max/avg(reading), "
                        f"{wl['rows']} rows/GPU, {wl['groups']} groups/GPU, {BATCH_ROWS}-row batches"
                        f"{', filter ' + ' '.join(map(str, wl['filt'])) if wl['filt'] else ''}",
            "rows_per_gpu": wl["rows"], "groups_per_gpu": wl["groups"], "batch_rows": BATCH_ROWS, "window_ms": wl["window_ms"],
            "slide_ms": wl["slide_ms"], "parallelism": f"key-hash partitions x{world} (one operator per GPU, disjoint key sets, no data-path collective)",
            "l2": "inputs (>= 10x L2) are streamed once per step; no explicit flush needed"}


# ------------------------------------------------------------------------------------------------
def pinned_host_batches(d, wl, rows, rank, world):
    """Arrow RecordBatches of the canonical schema whose buffers live in page-locked memory from dnz_host_alloc."""
    import pyarrow as pa
    from oracle import lib as olib
    L, OL = d.lib(), olib()
    nb = rows // BATCH_ROWS
    maxlen = 36 if wl["uuid"] else 8 + len(str((wl["groups"] - 1) * world + rank))
    sizes = dict(ts=8 * BATCH_ROWS, val=8 * BATCH_ROWS, off=4 * (BATCH_ROWS + 1), kb=maxlen * BATCH_ROWS)
    stride = sum((v + 255) // 256 * 256 for v in sizes.values())
    base = L.dnz_host_alloc(stride * nb)
    if not base:
        raise MemoryError("dnz_host_alloc failed")
    barrier = pa.array(["no_barrier"] * BATCH_ROWS, pa.utf8())
    schema = d.canonical_schema()
    meta_fields = list(schema.field(3).type)
    batches, in_bytes = [], 0

    def fill(b):
        p = base + b * stride
        a_ts, a_val = p, p + 8 * BATCH_ROWS
        a_off = a_val + 8 * BATCH_ROWS
        a_kb = (a_off + 4 * (BATCH_ROWS + 1) + 255) // 256 * 256
        used = OL.orc_synth_fill(b * BATCH_ROWS, BATCH_ROWS, 42 + rank, wl["groups"], wl["rows_per_ms"], T0, 1 if wl["uuid"] else 0,
                                 world, rank, a_ts, a_val, a_off, a_kb)
        return a_ts, a_val, a_off, a_kb, used
    # generate with a few threads (ctypes releases the GIL)
    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(max_workers=min(32, os.cpu_count() or 1)) as ex:
        addrs = list(ex.map(fill, range(nb)))
    keep = (L, base)
    for a_ts, a_val, a_off, a_kb, used in addrs:
        fb = lambda a, n: pa.foreign_buffer(a, n, base=keep)
        ts = pa.Array.from_buffers(pa.timestamp("ms"), BATCH_ROWS, [None, fb(a_ts, 8 * BATCH_ROWS)])
        occ = pa.Array.from_buffers(pa.int64(), BATCH_ROWS, [None, fb(a_ts, 8 * BATCH_ROWS)])
        val = pa.Array.from_buffers(pa.float64(), BATCH_ROWS, [None, fb(a_val, 8 * BATCH_ROWS)])
        key = pa.Array.from_buffers(pa.utf8(), BATCH_ROWS, [None, fb(a_off, 4 * (BATCH_ROWS + 1)), fb(a_kb, max(used, 1))])
        meta = pa.StructArray.from_arrays([barrier, ts], fields=meta_fields)
        batches.append(pa.RecordBatch.from_arrays([occ, val, key, meta], schema=schema))
        in_bytes += 20 * BATCH_ROWS + 4 + used
    return batches, in_bytes, base, addrs


def export_all(d, batches):
    """Pre-export RecordBatches to Arrow C-Data structs (binding overhead, outside the timed region)."""
    arr = (d.capi.ArrowArrayC * len(batches))()
    for i, b in enumerate(batches):
        b._export_to_c(C.addressof(arr[i]))
    return arr


# ------------------------------------------------------------------------------------------------
# parity of the timed legs (outside the timed regions): the rows a leg emitted for the windows that lie completely inside the
# first `sample` rows of its stream are compared, row by row, with the CPU oracle run over exactly those rows
def parity_sample_rows(wl, world):
    n = min(200_000_000 if world == 1 else 100_000_000, wl["rows"])
    return max(BATCH_ROWS, n // BATCH_ROWS * BATCH_ROWS)


def batches_from_addresses(addrs, n_batches):
    """oracle.Batch views over the page-locked buffers the e2e leg feeds to the operator (no copy)."""
    from oracle import Batch

    def view(addr, dt, n):
        return np.ctypeslib.as_array(C.cast(addr, C.POINTER(C.c_uint8)), shape=(n * np.dtype(dt).itemsize,)).view(dt)
    out = []
    for a_ts, a_val, a_off, a_kb, used in addrs[:n_batches]:
        out.append(Batch(ts=view(a_ts, np.int64, BATCH_ROWS), val=view(a_val, np.float64, BATCH_ROWS), key_off=view(a_off, np.int32, BATCH_ROWS + 1),
                         key_bytes=view(a_kb, np.uint8, max(used, 1))))
    return out


def oracle_sample(wl, batches, sample_rows):
    """Oracle rows (pyarrow Table) of the windows that end at or before the last full millisecond of the sample."""
    import pyarrow.compute as pc
    from tests.helpers import oracle_mt_arrays, result_table, rows_to_batch
    span_ms = sample_rows // wl["rows_per_ms"]                      # rows [0, span_ms * rows_per_ms) carry ts < T0 + span_ms
    cut = T0 + span_ms
    feed = list(batches) + [rows_to_batch([(cut + 2 * wl["window_ms"] + 1000, 1.0, b"sentinel")])]
    t = time.perf_counter()
    arr = oracle_mt_arrays(feed, wl["window_ms"], wl["slide_ms"], wl["filt"])
    dt = time.perf_counter() - t
    tab = result_table(arr, "w")
    tab = tab.filter(pc.less_equal(pc.add(tab["ws"], wl["window_ms"]), cut))
    return tab, cut, dt


class StepCapture(list):
    """The device results a step emits, copied on the operator's stream as each one is handed out (a result is valid only until
    the next call on the operator), into a buffer of `reserve` bytes allocated up front (beyond it, into fresh allocations).
    Capturing a timed step this way adds device-to-device copies to it but no host wait and, while the buffer lasts, no
    allocation; `to_host()` reads the copies back afterwards as `fetch_device_result`-style dicts."""
    FIELDS = {"key_off": np.int32, "key_valid": np.uint8, "agg_valid": np.uint8, "count": np.int64, "min": np.float64, "max": np.float64,
              "avg": np.float64, "window_start_ms": np.int64, "window_end_ms": np.int64}

    class _DeviceBytes:
        def __init__(self, ptr, n):
            self.__cuda_array_interface__ = {"shape": (n,), "typestr": "|u1", "data": (ptr, False), "version": 2}

    def __init__(self, torch, stream, device, reserve):
        super().__init__()
        self.torch, self.stream, self.device = torch, stream, device
        self.buf, self.used = torch.empty(reserve, dtype=torch.uint8, device=device), 0

    def take(self, w, r):
        t = self.torch

        def copy(ptr, n):
            if self.used + n <= self.buf.numel():
                dst = self.buf[self.used:self.used + n]
                self.used += (n + 255) // 256 * 256
            else:
                dst = t.empty(n, dtype=t.uint8, device=self.device)
            return dst.copy_(t.as_tensor(self._DeviceBytes(ptr, n), device=self.device), non_blocking=True) if n else dst
        with t.cuda.stream(self.stream):
            part = {f: copy(getattr(r, f), r.n_rows * np.dtype(dt).itemsize) for f, dt in self.FIELDS.items()}
            part["key_bytes"] = copy(r.key_bytes, r.key_bytes_len)
        self.append((r.key_bytes_len, part))

    def to_host(self):
        self.stream.synchronize()
        out = []
        for kb_len, part in self:
            h = {f: part[f].cpu().numpy().view(dt) for f, dt in self.FIELDS.items()}
            out.append({"key_off": np.append(h["key_off"], np.int32(kb_len)), "key_bytes": part["key_bytes"].cpu().numpy(),
                        "key_valid": h["key_valid"], "agg_valid": h["agg_valid"], "count": h["count"], "min": h["min"], "max": h["max"],
                        "avg": h["avg"], "window_start": h["window_start_ms"], "window_end": h["window_end_ms"]})
        return out


DUMP_ROWS = 1_000_000        # 7 float64 columns of this many rows: 56 MB per dump


def dump_outputs(out_dir, parts, seed=0):
    """Writes the rows of a step's device results (`fetch_device_result` dicts) as float64 arrays DIR/<column>.npy: window_start_ms,
    window_end_ms, key_id, count, min, max, avg, sorted by (window start, key).  key_id is the key's rank among the distinct keys
    of the step (-1 for a NULL key); min / max / avg are NaN where the aggregate is NULL.  Above DUMP_ROWS rows, a seeded sample
    of row positions in that order is written, so two builds that emit the same rows write the same sample."""
    import pyarrow as pa
    import pyarrow.compute as pc
    tabs = []
    for p in parts:
        n = len(p["count"])
        if not n:
            continue
        keys = pa.Array.from_buffers(pa.binary(), n, [None, pa.py_buffer(p["key_off"]), pa.py_buffer(p["key_bytes"])])
        keys = pc.if_else(pa.array(np.asarray(p["key_valid"]) != 0), keys, pa.scalar(None, pa.binary()))
        null = np.asarray(p["agg_valid"]) == 0
        tabs.append(pa.table({"window_start_ms": p["window_start"], "window_end_ms": p["window_end"], "key": keys, "count": p["count"],
                              **{c: np.where(null, np.nan, np.asarray(p[c], np.float64)) for c in ("min", "max", "avg")}}))
    cols = {"window_start_ms": pa.int64(), "window_end_ms": pa.int64(), "key": pa.binary(), "count": pa.int64(), "min": pa.float64(),
            "max": pa.float64(), "avg": pa.float64()}
    tab = pa.concat_tables(tabs) if tabs else pa.schema(cols).empty_table()
    tab = tab.sort_by([("window_start_ms", "ascending"), ("key", "ascending")])
    keys = pc.dictionary_encode(tab["key"].combine_chunks())
    rank = np.full(len(keys.dictionary) + 1, -1.0)                  # the last entry stands for the NULL key
    rank[pc.sort_indices(keys.dictionary).to_numpy()] = np.arange(len(keys.dictionary))
    out = {c: tab[c].to_numpy().astype(np.float64) for c in cols if c != "key"}
    out["key_id"] = rank[keys.indices.fill_null(len(keys.dictionary)).to_numpy()]
    pick = np.arange(tab.num_rows)
    if tab.num_rows > DUMP_ROWS:
        pick = np.sort(np.random.default_rng(seed).choice(tab.num_rows, DUMP_ROWS, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a[pick])
    return tab.num_rows, len(pick)


def plan_e2e_steps(fit, warmup, steps, n_parity_ops):
    """How many warm-up and timed e2e steps run when `fit` operators (one per step, plus the parity pass) fit into device memory:
    at most 3 warm-ups and `steps` timed steps, never fewer than one of each."""
    e_warm = min(warmup, 3, max(1, fit - 1 - n_parity_ops))
    e_steps = max(1, min(steps, fit - e_warm - n_parity_ops))
    return e_warm, e_steps


class Capture(list):
    """Collects a leg's emitted results, keeping only the polls that contain rows of windows ending at or before `cut`."""

    def __init__(self, cut, window_ms):
        super().__init__()
        self.cut, self.window_ms = cut, window_ms

    def take(self, w, r):
        self.append(w.fetch_device_result(r, max_keys=0))

    def append(self, part):
        if isinstance(part, dict):
            ws = np.asarray(part["window_start"])
            keep = len(ws) and int(ws.min()) + self.window_ms <= self.cut
        else:
            import pyarrow.compute as pc
            keep = part.num_rows and pc.min(part.column("window_start_time").cast("int64")).as_py() + self.window_ms <= self.cut
        if keep:
            super().append(part)


def leg_checksum(parts, cut, window_ms):
    """Order-independent checksum of the emitted rows of the windows that end at or before `cut`:
    (rows, sum of counts, xor of min bit patterns, xor of max bit patterns, sum of averages)."""
    n, sc, xmn, xmx, sa = 0, 0, 0, 0, 0.0
    for p in parts:
        if not len(p["count"]):
            continue
        m = (np.asarray(p["window_start"]) + window_ms) <= cut
        ok = m & ((np.asarray(p["agg_isnull"]) == 0) if "agg_isnull" in p else (np.asarray(p["agg_valid"]) != 0))
        n += int(m.sum()); sc += int(np.asarray(p["count"])[m].sum())
        xmn ^= int(np.bitwise_xor.reduce(np.asarray(p["min"], np.float64)[ok].view(np.uint64))) if ok.any() else 0
        xmx ^= int(np.bitwise_xor.reduce(np.asarray(p["max"], np.float64)[ok].view(np.uint64))) if ok.any() else 0
        sa += float(np.asarray(p["avg"], np.float64)[ok].sum())
    return (n, sc, xmn, xmx, sa)


def combine_checksums(cs):
    n = sum(c[0] for c in cs); sc = sum(c[1] for c in cs); sa = sum(c[4] for c in cs)
    xmn = xmx = 0
    for c in cs:
        xmn ^= c[2]; xmx ^= c[3]
    return (n, sc, xmn, xmx, sa)


def compare_with_oracle(got_parts, want, cut, wl, what):
    """got_parts: column-array dicts (device results) or pyarrow RecordBatches (Arrow results) of a leg."""
    import pyarrow as pa
    import pyarrow.compute as pc
    from tests.helpers import assert_tables_equal, concat_arrays, result_table
    tabs = []
    for p in got_parts:
        if isinstance(p, dict):
            if not len(p["count"]):
                continue
            t = result_table(concat_arrays([p]), "g")
        else:
            if p.num_rows == 0:
                continue
            nulls = pc.is_null(p.column("min"))
            t = pa.table({"ws": p.column("window_start_time").cast(pa.int64()), "key": p.column(0).cast(pa.binary()),
                          "count_g": p.column("count"),
                          "min_g": pa.array(p.column("min").fill_null(0.0).to_numpy(zero_copy_only=False).view(np.int64)),
                          "max_g": pa.array(p.column("max").fill_null(0.0).to_numpy(zero_copy_only=False).view(np.int64)),
                          "avg_g": p.column("average").fill_null(0.0), "null_g": nulls})
        tabs.append(t.filter(pc.less_equal(pc.add(t["ws"], wl["window_ms"]), cut)))
    got = pa.concat_tables(tabs) if tabs else want.slice(0, 0).rename_columns(["ws", "key", "count_g", "min_g", "max_g", "avg_g", "null_g"])
    n = assert_tables_equal(got, want)
    return {"leg": what, "rows_compared": int(n)}


_JSON_OUT = None


def claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries print there too (NCCL's version banner, for one), so fd 1 is pointed at
    stderr for the whole run and the JSON line goes to a private duplicate of the original stdout."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)
    return _JSON_OUT


def main():
    args = parse_args()
    claim_stdout()
    wl = dict(WORKLOADS[args.workload])
    if args.rows:
        wl["rows"] = args.rows
    if args.impl == "reference":
        run_reference(args, wl)
        return

    import torch
    import torch.distributed as dist
    import denormalized_b200 as d

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torchrun --nproc-per-node N for --gpus N")
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs writes the output of one operator: run it with --gpus 1")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback exists)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    L = d.lib()
    stream = torch.cuda.Stream(device=local)      # a non-blocking stream of its own: the legacy default stream synchronises with every blocking stream of the process (NCCL, torch)
    rows, G = wl["rows"], wl["groups"]
    last_ts = T0 + (rows - 1) // wl["rows_per_ms"]
    close_wm = (last_ts // 1000 + 1) * 1000 + 2 * wl["window_ms"]

    # ---- device-resident input: every rank owns a disjoint key set (key id * world + rank), same window structure
    dev = d.DeviceBatches(rows, BATCH_ROWS, seed=42 + rank, groups=G, rows_per_ms=wl["rows_per_ms"], uuid_keys=wl["uuid"], device=local,
                          key_mul=world, key_add=rank)

    def new_window(flags=0):
        return d.GpuStreamingWindow(d.canonical_schema(), "sensor_name", AGGS, wl["window_ms"], wl["slide_ms"], wl["filt"], device=local,
                                    flags=flags | args.flags, expected_groups=G, max_rows_per_launch=args.max_rows_per_launch,
                                    cuda_stream=stream.cuda_stream)

    GROUP = int(os.environ.get('DNZ_BENCH_GROUP', '1024'))       # batches (64 Mi rows) pushed between polls: emitted windows are consumed as the stream advances

    def step_device(w, capture=None):
        """One pass over the device-resident stream.  Batches are pushed 64 Mi rows at a time; the operator pipelines them (tile scan
        of group g+1 | aggregate + emission of group g | verification of group g-1) and the emitted windows are consumed as the
        stream advances with the non-forcing poll, so the host never waits between two kernels."""
        n_out = 0
        for g0 in range(0, dev.n_batches, GROUP):
            n = min(GROUP, dev.n_batches - g0)
            w.push_device(array=C.cast(C.byref(dev.array, g0 * C.sizeof(d.capi.DeviceBatchC)), C.POINTER(d.capi.DeviceBatchC)), n=n)
            while True:
                r = w.poll_device_ready()
                if r.n_rows == 0:
                    break
                n_out += r.n_rows
                if capture is not None:
                    capture.take(w, r)
        # close the remaining windows a few at a time: one poll must stay below 2 GiB of key bytes (Utf8 offsets are 32-bit),
        # which 10 M 36-byte keys x 12 open sliding windows (cfg 5) would exceed
        step_ms = max(wl["slide_ms"] or wl["window_ms"], 1000) * (1 if G >= 4_000_000 else 64)
        wm = (last_ts // 1000) * 1000
        while wm < close_wm:
            wm = min(wm + step_ms, close_wm)
            w.flush(wm)
            while True:
                r = w.poll_device()
                if r.n_rows == 0:
                    break
                n_out += r.n_rows
                if capture is not None:
                    capture.take(w, r)
        return n_out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def log(msg):
        if rank == 0:
            print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)
    log(f"device input ready: {rows} rows, {dev.n_batches} batches, {dev.algorithmic_bytes / 1e9:.2f} GB algorithmic")
    out_rows = 0
    for _ in range(args.warmup):
        w = new_window(); out_rows = step_device(w); w.close()
    # operators are created before the timed region (creation = allocation); huge tables (>= 4 M groups: tens of GB per
    # operator) are created one at a time instead, from the memory the previous one returned to the pool
    lazy = G >= 4_000_000
    wins = [None if lazy else new_window(d.capi.FLAG_KERNEL_TIMING) for _ in range(args.steps)]
    stats = []
    dumped = None               # what the last timed step emits; room for ~4x the warm-up's rows (a poll re-reads its set's keys)
    if args.dump_outputs:
        room = 4 * out_rows * (len(StepCapture.FIELDS) * 8 + 40) + (64 << 20)
        dumped = StepCapture(torch, stream, local, min(room, torch.cuda.mem_get_info()[0] // 4))
    sampler = ClockSampler(local); sampler.start()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for i, w in enumerate(wins):
        if lazy:
            w = new_window(d.capi.FLAG_KERNEL_TIMING)
        step_device(w, dumped if i == args.steps - 1 else None)
        if lazy:
            stats.append(w.stats()); w.close()
    ev1.record(stream)
    barrier()
    clocks = sampler.stop()
    ms = ev0.elapsed_time(ev1)
    if world > 1:
        allms = [None] * world
        dist.all_gather_object(allms, round(ms / args.steps, 2))
        log(f"device-resident ms/step per rank: {allms}")
    log(f"device-resident: {ms / args.steps:.2f} ms/step")
    if dumped is not None:
        n_rows, n_dumped = dump_outputs(args.dump_outputs, dumped.to_host())
        del dumped
        log(f"last timed step: {n_rows} rows emitted, {n_dumped} written to {args.dump_outputs}")
    if not lazy:
        stats = [w.stats() for w in wins]
        for w in wins:
            w.close()
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = rows * world * args.steps / (ms * 1e-3)
    parity = []
    want = cut = None
    if not args.no_parity:
        from tests.helpers import host_stream
        ps = parity_sample_rows(wl, world)
        hs = host_stream(ps, groups=G, rows_per_ms=wl["rows_per_ms"], uuid_keys=wl["uuid"], seed=42 + rank, key_mul=world, key_add=rank)
        want, cut, odt = oracle_sample(wl, hs, ps)
        del hs
        log(f"oracle over the first {ps} rows of this rank's stream: {odt:.1f} s, {want.num_rows} rows in complete windows")
        capd = Capture(cut, wl["window_ms"])
        wv = new_window(); step_device(wv, capd); wv.close()
        parity.append(compare_with_oracle(capd, want, cut, wl, "value"))
        del capd
        log("value leg: emitted rows equal the oracle's")
    agg_ms = sum(s["agg_kernel_ms"] for s in stats); agg_bytes = sum(s["agg_algorithmic_bytes"] for s in stats)
    agg_launches = sum(s["agg_launches"] for s in stats); launches = sum(s["total_launches"] for s in stats)
    peak, peak_src = measured_peak()
    achieved = agg_bytes / (agg_ms * 1e-3) / 1e9 if agg_ms > 0 else 0.0
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "agg_kernel_traffic.json")) as f:
            traffic = json.load(f).get("dram_bytes_per_launch")
    except Exception:
        pass

    # ---- N>1 only: the same stream NOT key-partitioned -- every rank sees every key, batches are dealt to ranks, and the
    # closed panes' partial states meet at their owners through ONE all-to-all per exchange step (NCCL over NVLink):
    # RepartitionExec(Hash) replaced by the pane exchange (denormalized_b200/exchange.py).  Reported beside `value`.
    exchange = None
    if world > 1 and not args.no_exchange:
        from denormalized_b200 import ExchangeGroup
        dev.free()
        devx = d.DeviceBatches(rows, BATCH_ROWS, seed=42 + rank, groups=G, rows_per_ms=wl["rows_per_ms"], uuid_keys=wl["uuid"], device=local)
        endm = d.DeviceBatches(1, 1, seed=7, groups=1, rows_per_ms=1, t0_ms=close_wm, device=local)     # end-of-stream marker row

        def rendezvous(blob):        # the one thing the library asks of its host: an all-gather of a few hundred bytes at creation
            t = torch.frombuffer(bytearray(blob), dtype=torch.uint8).cuda()
            out = torch.empty(world * t.numel(), dtype=torch.uint8, device="cuda")
            dist.all_gather_into_tensor(out, t)
            raw = out.cpu().numpy().tobytes()
            return [raw[i * len(blob):(i + 1) * len(blob)] for i in range(world)]
        # one packet per (closed pane, group) a rank holds for a key owned elsewhere: size the receive rings for one step
        XSTEP = int(os.environ.get('DNZ_BENCH_XSTEP', '2'))          # superbatches (64 Mi rows each) per exchange step
        panes_per_step = max(2, (XSTEP * GROUP * BATCH_ROWS) // max(1, wl["rows_per_ms"] * (wl["slide_ms"] or wl["window_ms"])) + 2)
        ring_entries = int(min(1 << 30, max(1 << 20, 1.25 * min(G, XSTEP * GROUP * BATCH_ROWS) * panes_per_step)))
        grp = ExchangeGroup.create(rank, world, local, rendezvous, ring_entries=ring_entries,
                                   ring_key_bytes=int(min((1 << 31) - 4096, ring_entries * (40 if wl["uuid"] else 16))))

        def step_exchange(w, capture=None):
            def take(r):
                if capture is not None and r.n_rows:
                    capture.append(w.fetch_device_result(r, max_keys=0))
                return r.n_rows
            for gi, g0 in enumerate(range(0, devx.n_batches, GROUP)):
                n = min(GROUP, devx.n_batches - g0)
                w.push_device(array=C.cast(C.byref(devx.array, g0 * C.sizeof(d.capi.DeviceBatchC)), C.POINTER(d.capi.DeviceBatchC)), n=n)
                if gi % XSTEP == XSTEP - 1:
                    grp.step(w)                                 # COLLECTIVE: global watermark, pack -> peers' rings, merge, emit (nothing waited for)
                while take(w.poll_device_ready()):
                    pass
            w.push_device(endm)
            grp.flush(w)                                        # end of stream: process + three steps (publish | pack | merge + emit)
            while take(w.poll_device()):
                pass
            return w.stats()["rows_out"]

        def xwindow():
            w = new_window(d.capi.FLAG_KERNEL_TIMING); grp.attach(w); return w
        xo = 0
        for _ in range(max(1, args.warmup - 1)):
            w = xwindow(); xo = step_exchange(w); x_base = w.stats()["exchanged_out"]; w.close()
        xw = [xwindow() for _ in range(args.steps)]
        barrier()
        x0, x1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        x0.record(stream)
        for w in xw:
            xo = step_exchange(w)
        x1.record(stream)
        barrier()
        allx = [None] * world
        dist.all_gather_object(allx, round(x0.elapsed_time(x1) / args.steps, 2))
        log(f"exchange ms/step per rank: {allx}")
        tx = torch.tensor([x0.elapsed_time(x1)], dtype=torch.float64, device="cuda"); dist.all_reduce(tx, op=dist.ReduceOp.MAX)
        to = torch.tensor([xo], dtype=torch.int64, device="cuda"); dist.all_reduce(to)
        xs = [w.stats() for w in xw]
        tp = torch.tensor([xs[-1]["exchanged_out"] - x_base], dtype=torch.int64, device="cuda"); dist.all_reduce(tp)     # the counter belongs to the group (cumulative)
        for w in xw:
            w.close()
        xms = float(tx.item())
        xagg_ms = sum(s_["agg_kernel_ms"] for s_ in xs); xagg_bytes = sum(s_["agg_algorithmic_bytes"] for s_ in xs)
        exchange = {"value": rows * world * args.steps / (xms * 1e-3), "unit": "rows/s", "ms_per_step": xms / args.steps,
                    "rows_out_per_step": int(to.item()), "packets_per_step": int(tp.item()) // args.steps,
                    "nvlink_bytes_per_step": int(tp.item()) // args.steps * 80,
                    "agg_kernel_ms": xagg_ms, "agg_algorithmic_bytes": xagg_bytes, "agg_launches": sum(s_["agg_launches"] for s_ in xs),
                    "launches": sum(s_["total_launches"] for s_ in xs),
                    "what": f"{rows} rows/GPU of ONE {G}-key stream dealt to {world} GPUs (NOT key-partitioned: every rank sees every key); "
                            f"per {XSTEP * 64} Mi rows/GPU one fused exchange step of the library-owned communicator (dnz_group): global watermark, "
                            "closed panes' partial states packed by owner = key hash % world and written straight into the owners' "
                            "receive rings over NVLink (remote-atomic reservation + P2P stores, interprocess CUDA events), owner merge, "
                            "owners emit; no NCCL / host copy in the data path"}
        if not args.no_parity:
            # every rank owns a share of the keys: order-independent checksums of the rows each rank emitted for the windows inside
            # the sample are combined on rank 0 and compared with the oracle run over the interleaved sample streams of ALL ranks
            psx = max(BATCH_ROWS, min(rows, 200_000_000 // world) // BATCH_ROWS * BATCH_ROWS)
            cutx = T0 + psx // wl["rows_per_ms"]
            capx = Capture(cutx, wl["window_ms"])
            w = xwindow(); xo_fresh = step_exchange(w, capx); w.close()
            mine = leg_checksum(capx, cutx, wl["window_ms"])
            # the timed streams ran through operators attached long before their stream began: they must emit what this one did
            tfresh = torch.tensor([xo_fresh], dtype=torch.int64, device="cuda"); dist.all_reduce(tfresh)
            exchange["rows_out_fresh_operator"] = int(tfresh.item())
            exchange["rows_out_consistent"] = int(tfresh.item()) == int(to.item())
            if not exchange["rows_out_consistent"]:
                log(f"exchange leg: the timed streams emitted {int(to.item())} rows per step, a fresh operator {int(tfresh.item())} -- the timed figure is NOT valid")
            del capx
            allsums = [None] * world
            dist.all_gather_object(allsums, mine)
            if rank == 0:
                from tests.helpers import host_stream, oracle_mt_arrays, rows_to_batch
                per_rank = [host_stream(psx, groups=G, rows_per_ms=wl["rows_per_ms"], uuid_keys=wl["uuid"], seed=42 + r) for r in range(world)]
                feed = [per_rank[r][i] for i in range(len(per_rank[0])) for r in range(world)]      # batch i of every rank, then batch i+1 ...
                feed.append(rows_to_batch([(cutx + 2 * wl["window_ms"] + 1000, 1.0, b"sentinel")]))
                oarr = oracle_mt_arrays(feed, wl["window_ms"], wl["slide_ms"], wl["filt"])
                del feed, per_rank
                ref = leg_checksum([oarr], cutx, wl["window_ms"])
                got = combine_checksums(allsums)
                assert got[:4] == ref[:4], f"exchange leg differs from the oracle: {got} != {ref}"
                assert abs(got[4] - ref[4]) <= 1e-9 * abs(ref[4]), f"exchange leg: sum of averages {got[4]} != {ref[4]}"
                parity.append({"leg": "exchange", "rows_compared": int(ref[0]), "how": "checksums: rows, sum(count), xor(min bits), xor(max bits), sum(avg) 1e-9"})
                log("exchange leg: checksums of the emitted rows equal the oracle's")
        devx.free(); endm.free(); grp.close()
        log(f"exchange leg: {xms / args.steps:.2f} ms/step")

    # ---- e2e: host Arrow buffers (pinned) through dnz_window_push / dnz_window_poll
    e2e = None
    if not args.no_e2e:
        free_gb = 64.0
        try:
            import psutil
            free_gb = psutil.virtual_memory().available / 2**30
        except Exception:
            pass
        # the whole stream when the host has the memory for it (40 B/row pinned), else its first 256 Mi rows
        cap = rows if free_gb / world > 6 * rows * 40 / 2**30 else 268_435_456
        e2e_rows = args.e2e_rows or int(min(rows, cap, max(BATCH_ROWS, (free_gb / 4 / world) * 2**30 / 40)))
        e2e_rows = max(BATCH_ROWS, e2e_rows // BATCH_ROWS * BATCH_ROWS)
        hb, in_bytes, base, hb_addrs = pinned_host_batches(d, wl, e2e_rows, rank, world)
        e_last = T0 + (e2e_rows - 1) // wl["rows_per_ms"]
        e_close = (e_last // 1000 + 1) * 1000 + 2 * wl["window_ms"]
        launch_rows = args.max_rows_per_launch or (64 << 20)
        reserve_bytes = int(min(launch_rows, e2e_rows) * (in_bytes / e2e_rows) * 1.05) + (64 << 20)
        # Every e2e step runs through its own operator, created (and its device staging reserved) before the timed region: three
        # superbatches in flight x `reserve_bytes` of staging + the deferred-row lists + results ~ 9 GB per operator for cfg 2.
        # The number of e2e steps is therefore bounded by the free device memory (the device-resident input of the other legs is
        # released first); `e2e.steps` / `e2e.warmup` say what was run.
        dev.free()
        torch.cuda.synchronize()
        free_dev = torch.cuda.mem_get_info()[0]
        per_op = 3 * reserve_bytes + 3 * min(launch_rows, max(e2e_rows, 1 << 20)) * 8 + (3 << 29)
        fit = max(3, int(free_dev * 0.85) // per_op)
        if world > 1:           # every rank runs the same number of steps
            tf = torch.tensor([fit], dtype=torch.int64, device="cuda")
            dist.all_reduce(tf, op=dist.ReduceOp.MIN)
            fit = int(tf.item())
        n_parity_ops = 0 if args.no_parity else 1
        e_warm, e_steps = plan_e2e_steps(fit, args.warmup, args.steps, n_parity_ops)
        n_e2e_steps = e_warm + e_steps
        n_e2e_total = n_e2e_steps + n_parity_ops                      # + one untimed pass whose output is compared with the oracle
        log(f"e2e: {free_dev / 2**30:.0f} GiB of device memory free, ~{per_op / 2**30:.1f} GiB per operator -> {e_warm} warm-up + {e_steps} timed steps")
        exported = [export_all(d, hb) for _ in range(n_e2e_total)]
        e_wins = [new_window() for _ in range(n_e2e_total)]
        for w_ in e_wins:       # operator start-up (device staging for host batches) belongs to creation, not to the stream
            w_.reserve_input(reserve_bytes)
        ca, cs, has = d.capi.ArrowArrayC(), d.capi.ArrowSchemaC(), C.c_int32(0)
        push, poll, poll_ready, flush = L.dnz_window_push, L.dnz_window_poll, L.dnz_window_poll_ready, L.dnz_window_flush
        rel = C.CFUNCTYPE(None, C.c_void_p)

        def step_host(i, capture=None):
            h = e_wins[i]._h
            arr = exported[i]
            n_out = 0
            for k in range(len(hb)):
                rc = push(h, C.byref(arr[k]))
                if rc:
                    raise d.DnzError(rc, L.dnz_window_last_error(h).decode())
                last = k == len(hb) - 1
                if last or (k + 1) % GROUP == 0:      # consume emitted windows as the stream advances
                    if last:
                        rc = flush(h, e_close) or poll(h, C.byref(ca), C.byref(cs), C.byref(has))
                    else:       # hand over what has been emitted so far; queued batches keep streaming
                        rc = poll_ready(h, C.byref(ca), C.byref(cs), C.byref(has))
                    if rc:
                        raise d.DnzError(rc, L.dnz_window_last_error(h).decode())
                    n_out += ca.length
                    if capture is not None:      # takes ownership of both structs
                        import pyarrow as pa
                        capture.append(pa.RecordBatch._import_from_c(C.addressof(ca), C.addressof(cs)))
                    else:
                        rel(ca.release)(C.addressof(ca)); rel(cs.release)(C.addressof(cs))
            return n_out
        log(f"e2e host batches ready: {e2e_rows} rows")
        for i in range(e_warm):
            step_host(i)
        d2h0 = sum(w.stats()["d2h_bytes"] for w in e_wins)
        barrier()
        t0 = time.perf_counter()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(e_warm, n_e2e_steps):
            e_out = step_host(i)
        e1.record(stream)
        barrier()
        wall = time.perf_counter() - t0
        ems = max(e0.elapsed_time(e1), wall * 1e3 * 0.0)   # device clock; the wall clock is reported beside it
        te = torch.tensor([ems, wall * 1e3], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        ems, wall_ms = float(te[0].item()), float(te[1].item())
        d2h = (sum(w.stats()["d2h_bytes"] for w in e_wins[:n_e2e_steps]) - d2h0) // e_steps
        h2d = e_wins[n_e2e_steps - 1].stats()["h2d_bytes"]
        pageable = e_wins[n_e2e_steps - 1].stats()["h2d_pageable_bytes"]
        if not args.no_parity:
            if e2e_rows < parity_sample_rows(wl, world):     # shorter host stream than the oracle sample: its own oracle run
                want, cut, odt = oracle_sample(wl, batches_from_addresses(hb_addrs, e2e_rows // BATCH_ROWS), e2e_rows)
            cap = Capture(cut, wl["window_ms"])
            step_host(n_e2e_total - 1, cap)
            parity.append(compare_with_oracle(cap, want, cut, wl, "e2e"))
            del cap
            log("e2e leg: emitted rows equal the oracle's")
        for w in e_wins:
            w.close()
        # ---- the same call sequence with PAGEABLE Arrow buffers (what arrow-rs hands over when the decoder does not allocate
        # through dnz_host_alloc): the library falls back to cudaMemcpyAsync, which the driver stages through its own pinned buffers
        pageable_e2e = None
        if rank == 0 or world > 1:
            import pyarrow as pa
            p_rows = min(e2e_rows, 134_217_728) // BATCH_ROWS * BATCH_ROWS
            p_nb = p_rows // BATCH_ROWS
            schema = d.canonical_schema(); meta_fields = list(schema.field(3).type)
            barrier_col = pa.array(["no_barrier"] * BATCH_ROWS, pa.utf8())
            pbatches = []
            for hbv in batches_from_addresses(hb_addrs, p_nb):          # numpy copies of the pinned buffers = ordinary heap memory
                ts_b, val_b = pa.py_buffer(hbv.ts.copy()), pa.py_buffer(hbv.val.copy())
                off_b, kb_b = pa.py_buffer(hbv.key_off.copy()), pa.py_buffer(hbv.key_bytes.copy())
                tsa = pa.Array.from_buffers(pa.timestamp("ms"), BATCH_ROWS, [None, ts_b])
                pbatches.append(pa.RecordBatch.from_arrays([pa.Array.from_buffers(pa.int64(), BATCH_ROWS, [None, ts_b]),
                                                            pa.Array.from_buffers(pa.float64(), BATCH_ROWS, [None, val_b]),
                                                            pa.Array.from_buffers(pa.utf8(), BATCH_ROWS, [None, off_b, kb_b]),
                                                            pa.StructArray.from_arrays([barrier_col, tsa], fields=meta_fields)], schema=schema))
            p_last = T0 + (p_rows - 1) // wl["rows_per_ms"]
            p_close = (p_last // 1000 + 1) * 1000 + 2 * wl["window_ms"]
            n_p = 1 + min(args.steps, 3)
            p_exp = [export_all(d, pbatches) for _ in range(n_p)]
            p_wins = [new_window() for _ in range(n_p)]
            for w_ in p_wins:
                w_.reserve_input(int(min(launch_rows, p_rows) * (in_bytes / e2e_rows) * 1.05) + (64 << 20))

            def step_pageable(i):
                h = p_wins[i]._h
                n_out = 0
                for k in range(p_nb):
                    rc = push(h, C.byref(p_exp[i][k]))
                    if rc:
                        raise d.DnzError(rc, L.dnz_window_last_error(h).decode())
                    last = k == p_nb - 1
                    if last or (k + 1) % GROUP == 0:
                        rc = (flush(h, p_close) or poll(h, C.byref(ca), C.byref(cs), C.byref(has))) if last else poll_ready(h, C.byref(ca), C.byref(cs), C.byref(has))
                        if rc:
                            raise d.DnzError(rc, L.dnz_window_last_error(h).decode())
                        n_out += ca.length
                        rel(ca.release)(C.addressof(ca)); rel(cs.release)(C.addressof(cs))
                return n_out
            step_pageable(0)
            barrier()
            tp0 = time.perf_counter()
            for i in range(1, n_p):
                step_pageable(i)
            barrier()
            p_wall = time.perf_counter() - tp0
            p_bytes = p_wins[-1].stats()["h2d_pageable_bytes"]
            for w_ in p_wins:
                w_.close()
            tpw = torch.tensor([p_wall], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(tpw, op=dist.ReduceOp.MAX)
            p_wall = float(tpw.item())
            pageable_e2e = {"value": p_rows * world * (n_p - 1) / p_wall, "unit": "rows/s", "rows_per_step": p_rows * world, "steps": n_p - 1,
                            "h2d_pageable_bytes_per_step": int(p_bytes), "gb_per_s": p_bytes * (n_p - 1) / p_wall / 1e9,
                            "sample": f"first {p_rows} rows/GPU of the stream in ordinary (pageable) heap memory: cudaMemcpyAsync path, wall clock"}
            del pbatches, p_exp
        e2e = {"value": e2e_rows * world * e_steps / (ems * 1e-3), "unit": "rows/s", "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(d2h), "rows_per_step": e2e_rows * world, "ms_per_step": ems / e_steps,
               "wall_ms_per_step": wall_ms / e_steps, "steps": e_steps, "warmup": e_warm,
               "rows_out_per_step": int(e_out), "pinned_fraction": 1.0 - pageable / max(h2d, 1),
               "h2d_gb_per_s": h2d / (ems / e_steps * 1e-3) / 1e9 / 1.0,
               "sample": f"first {e2e_rows} rows/GPU of the stream, Arrow buffers in pinned host memory (dnz_host_alloc)",
               "pageable": pageable_e2e}
        del hb, exported
        L.dnz_host_free(base)

    log("e2e done" if e2e else "e2e skipped")
    # ---- CPU baseline on the host cores (rank 0, N=1 only)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        threads = choose_threads(wl)
        crow = args.cpu_rows or auto_cpu_rows(wl, threads)
        rate, dt, n, _ = cpu_baseline(wl, crow, threads)
        cpu = {"value": rate, "unit": "rows/s", "cores": threads, "threads": threads, "host_cores": os.cpu_count(), "kind": "port",
               "sample": f"{n} rows ({n // BATCH_ROWS} batches) of the {args.workload} stream, {dt:.1f} s, oracle/ hash-partitioned over {threads} threads"}

    if rank == 0:
        line = {"metric": "rows/sec windowed group-agg on synthetic sensor batches", "value": value, "unit": "rows/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_config(args, wl, world),
                "rows_out_per_step": int(out_rows), "gpu_launches": int(launches), "clocks": clocks,
                "roofline": {"bound": "hbm", "kernel": "k_aggregate", "achieved": achieved, "peak": peak, "unit": "GB/s",
                             "frac": achieved / peak if peak else None, "traffic": traffic, "peak_source": peak_src,
                             "launches": int(agg_launches), "avg_launch_ms": agg_ms / max(agg_launches, 1),
                             "algorithmic_bytes_per_row": agg_bytes / max(rows * args.steps, 1)},
                "e2e": e2e, "cpu_baseline": cpu,
                "parity_checked": bool(parity) and not args.no_parity, "parity": parity}
        if exchange and not exchange.get("rows_out_consistent", True):
            # the timed exchange streams did not emit what a fresh operator emits on the same stream: that figure is not a measurement
            # of the path.  The key-partitioned leg (verified row by row) stays the headline; the exchange leg is kept with its flag.
            line["exchange"] = exchange
            line["config"]["note"] = "exchange leg rejected (rows_out_consistent false): headline = key-partitioned leg"
        elif exchange:
            # N > 1: the headline is the UN-PARTITIONED stream through the fused exchange; the key-partitioned run (no data-path
            # collective, keys generated pre-partitioned) is kept beside it
            line["partitioned"] = {"value": value, "unit": "rows/s", "ms_per_step": ms / args.steps,
                                   "what": "every rank aggregates its own hash partition of the key space (keys generated pre-partitioned, no exchange)",
                                   "roofline_frac": line["roofline"]["frac"], "gpu_launches": int(launches)}
            xa = exchange["agg_algorithmic_bytes"] / (exchange["agg_kernel_ms"] * 1e-3) / 1e9 if exchange["agg_kernel_ms"] > 0 else 0.0
            line.update({"value": exchange["value"], "ms_per_step": exchange["ms_per_step"], "rows_out_per_step": exchange["rows_out_per_step"],
                         "gpu_launches": int(exchange["launches"])})
            line["roofline"].update({"achieved": xa, "frac": xa / peak if peak else None, "launches": int(exchange["agg_launches"]),
                                     "avg_launch_ms": exchange["agg_kernel_ms"] / max(exchange["agg_launches"], 1),
                                     "algorithmic_bytes_per_row": exchange["agg_algorithmic_bytes"] / max(rows * args.steps, 1)})
            line["config"]["parallelism"] = (f"one stream of {G} keys dealt to {world} GPUs (not key-partitioned) + fused pane exchange over NVLink "
                                             "(dnz_group: P2P stores into the owners' rings, owner = key hash % world)")
            line["exchange"] = exchange
        print(json.dumps(line), file=claim_stdout(), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
