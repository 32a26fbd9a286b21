#!/usr/bin/env python
"""bench.py — decoded+aggregated points/s of the tskv scan hot path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            our arm (CUDA, one rank per GPU under torchrun)
  python bench.py --impl reference --steps K --warmup W    the reference algorithm on the host CPU cores
                                                           (oracle port: the Rust reference cannot be built here)
  python bench.py --workload C1|C2|C3|C4|C5 [--series n]   the other BASELINE shapes (default C4, the headline)
  python bench.py ... --dump-outputs DIR                   also write what the last timed step computed, DIR/<name>.npy
                                                           (inputs are seeded: the same arguments give the same inputs;
                                                           f64 sums / means may differ in the last bits between runs
                                                           as the device adds in varying order, compare within 1e-6)

Workload C4 (config.workload, the configuration BASELINE's metric is quoted on): 1 000 000 series x 1 000 points,
mixed i64 (Delta/simple8b) and f64 (Gorilla, full-mantissa) columns, 20 % of the series with jittered timestamps
(simple8b time pages), 1 % of the pages with 5 % nulls, tag predicate selecting 10 % of the series, GROUP BY 1-minute
bucket with count/sum/min/max/mean. Series are sharded in contiguous id ranges over N GPUs (strong scaling: total work
fixed); the only collective is the exchange of the per-bucket partials.

One JSON line on stdout (rank 0). A "step" is one full pass: series selection -> work list -> fused
decode/filter/bucket-reduce kernels -> (exchange) -> dense result.
  value     whole-job points/s with the pages already resident in HBM (device time, CUDA events, max over ranks);
            `value_crc_per_step` is the same with every page's CRC32 re-checked on the device every step (what the
            CPU arm and the reference do on every read)
  e2e       the same through the public call with the pages in HOST memory: query args H2D, PCIe gather of
            the selected pages, device CRC32, scan, result D2H (wall clock around synchronised calls, max over ranks)
  roofline  fused phase: encoded bytes it reads / its CUDA-event time vs the measured HBM copy peak
  cpu_baseline  the oracle (port of the reference algorithm) on the host cores: the WHOLE workload, every step
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from cnosdb_b200 import cabi, datagen  # noqa: E402
from cnosdb_b200.engine import PushedAggregate, QueryOption  # noqa: E402
from cnosdb_b200.parallel import select_tag_subset, shard_range  # noqa: E402

METRIC = "decoded+aggregated points/s"
W_NS = 60_000_000_000
AGGS = ["count", "sum", "min", "max", "mean"]
BIN_NAMES = {0: "ts=RLE,val=simple8b", 1: "ts=RLE,val=gorilla", 2: "ts=RLE,val=generic", 3: "ts=simple8b,val=simple8b",
             4: "ts=simple8b,val=gorilla", 5: "ts=simple8b,val=generic", 6: "ts=generic,val=simple8b",
             7: "ts=generic,val=gorilla", 8: "ts=generic,val=generic", 9: "ts=RLE,val=simple8b (<=1024 rows)",
             10: "ts=simple8b,val=simple8b (<=1024 rows)", 11: "ts=RLE,val=gorilla (<=1024 rows)",
             12: "ts=simple8b,val=gorilla (<=1024 rows)"}


def bucket_spec(width=W_NS, n_points=1000, slack=1_000_000):
    lo = datagen.TSBS_T0 - slack
    hi = datagen.TSBS_T0 + (n_points - 1) * datagen.TSBS_STEP + slack
    start = lo - (lo % width)
    return start, int((hi - start) // width + 1)


class Workload:
    """One BASELINE shape: how a shard is generated, which series are selected, the query."""

    def __init__(self, key, default_series, describe, gen_kw, select, query, n_points=1000, fields_per_series=1):
        self.key, self.default_series, self.describe = key, default_series, describe
        self.gen_kw, self.select, self.query = gen_kw, select, query
        self.n_points, self.fields_per_series = n_points, fields_per_series

    def generate(self, first, count):
        return datagen.generate(count, first_series_id=first, series_stride=1, n_points=self.n_points, **self.gen_kw)

    def config(self, n_series):
        sel = self.select(n_series)
        return {"workload": self.describe % n_series, "series_total": n_series, "points_per_series": self.n_points,
                "selected_series": int(n_series if sel is None else len(sel)),
                "sharding": "contiguous series-id ranges, one per GPU"}


def _q_c4(sel, **kw):
    fbs, nb = bucket_spec()
    return QueryOption([PushedAggregate(1, cabi.TSKV_PT_I64, AGGS), PushedAggregate(2, cabi.TSKV_PT_F64, AGGS)],
                       series_ids=sel, width=W_NS, first_bucket_start=fbs, n_buckets=nb, **kw)


def _q_c2(sel, **kw):  # closed range covering rows 250..749; per-series sum + count
    a = datagen.TSBS_T0 + 250 * datagen.TSBS_STEP
    b = datagen.TSBS_T0 + 749 * datagen.TSBS_STEP
    return QueryOption([PushedAggregate(1, cabi.TSKV_PT_F64, ["count", "sum"])], series_ids=sel, time_ranges=[(a, b)],
                       group_by_series=True, **kw)


def _q_c3(sel, **kw):
    fbs, nb = bucket_spec()
    return QueryOption([PushedAggregate(c, cabi.TSKV_PT_I64, ["mean", "max"]) for c in range(1, 11)], series_ids=sel,
                       width=W_NS, first_bucket_start=fbs, n_buckets=nb, **kw)


def _q_c5(sel, **kw):  # last hour (360 points): max per 5-minute bucket + last point, 5 fields
    w = 5 * W_NS
    fbs, nb = bucket_spec(width=w, n_points=360)
    return QueryOption([PushedAggregate(c, cabi.TSKV_PT_I64, ["max", "last"]) for c in range(1, 6)], series_ids=sel,
                       width=w, first_bucket_start=fbs, n_buckets=nb, **kw)


WORKLOADS = {
    "C4": Workload("C4", 1_000_000,
                   "C4: %d series x 1000 pts, mixed i64 Delta / f64 Gorilla, 20%% jittered ts, 1%% pages with 5%% nulls, "
                   "10%% tag selection, group by 1-min bucket (count,sum,min,max,mean)",
                   dict(n_fields=1, value_kind=datagen.MIXED, seed=4, jitter_permille=200, jitter_max=999_999,
                        null_page_permille=10, null_row_permille=50),
                   lambda n: select_tag_subset(n, 10), _q_c4),
    "C2": Workload("C2", 10_000,
                   "C2: %d series x 1000 f64 Gorilla points (walk + full-mantissa noise), closed time range over rows "
                   "250..749, sum + count per series",
                   dict(n_fields=1, value_kind=datagen.F64_NOISE, seed=2), lambda n: None, _q_c2),
    "C3": Workload("C3", 100_000,
                   "C3: TSBS devops cpu-only, %d hosts x 10 i64 fields x 1000 pts, mean + max per 1-min bucket over all hosts",
                   dict(n_fields=10, value_kind=datagen.I64_WALK, seed=3), lambda n: None, _q_c3, fields_per_series=10),
    "C5": Workload("C5", 10_000_000,
                   "C5: single-groupby-5-8-1 shape, %d series x 5 of 10 i64 fields, last hour (360 pts): max per 5-min "
                   "bucket + last point",
                   dict(n_fields=10, value_kind=datagen.I64_WALK, seed=5), lambda n: None, _q_c5, n_points=360,
                   fields_per_series=10),
}


def generate_shard(n_total, rank, world, workload="C4"):
    lo, hi = shard_range(n_total, rank, world)
    return WORKLOADS[workload].generate(lo, hi - lo)


def make_query(series_ids, workload="C4"):
    return WORKLOADS[workload].query(series_ids)


def concat_arenas(parts):
    """[(arena, descs), ...] -> one arena + descriptor table (page offsets rebased, 16-byte alignment kept)."""
    chunks, descs, base = [], [], 0
    for arena, d in parts:
        pad = (-base) % 16
        if pad:
            chunks.append(np.zeros(pad, dtype=np.uint8))
            base += pad
        dd = np.array(d, dtype=cabi.PAGE_DESC_DTYPE, copy=True)
        dd["offset"] += base
        descs.append(dd)
        chunks.append(np.asarray(arena))
        base += len(arena)
    return np.concatenate(chunks), np.concatenate(descs)


class ClockSampler:
    """SM clock / power / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe). The region is
    ~20 ms long, so NVML is polled from a thread every millisecond (what nvidia-smi reads, without its 100 ms period);
    `nvidia-smi -lms` is the fallback when pynvml is missing."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")
    REASON_BITS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
                   0x80: "hw_power_brake_slowdown"}

    def __init__(self, index):
        self.index, self.rows, self.proc, self.nvml, self.handle, self.stop_flag = index, [], None, None, None, False
        try:
            import pynvml
            pynvml.nvmlInit()
            handle = None
            try:
                import torch
                uuid = str(torch.cuda.get_device_properties(index).uuid)
                handle = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
            except Exception:
                handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.nvml, self.handle = pynvml, handle
        except Exception:
            self.nvml = None

    def start(self):
        if self.nvml:
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _poll(self):
        n, h = self.nvml, self.handle
        while not self.stop_flag:
            try:
                sm = n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM)
                mx = n.nvmlDeviceGetMaxClockInfo(h, n.NVML_CLOCK_SM)
                pw = n.nvmlDeviceGetPowerUsage(h) / 1000.0
                try:
                    rs = n.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    rs = n.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.rows.append((time.perf_counter(), float(sm), float(mx), pw, int(rs)))
            except Exception:
                pass
            time.sleep(0.001)

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self, t_begin=None, t_end=None):
        """t_begin / t_end (time.perf_counter): host-side bounds of the timed region; NVML samples outside are dropped."""
        if self.nvml:
            self.stop_flag = True
            self.thread.join(timeout=1.0)
            rows = [r for r in self.rows if (t_begin is None or r[0] >= t_begin) and (t_end is None or r[0] <= t_end)]
            if not rows:
                rows = self.rows[-3:]
            reasons = sorted({name for r in rows for bit, name in self.REASON_BITS.items() if r[4] & bit})
            return {"sm_mhz": float(np.median([r[1] for r in rows])) if rows else None,
                    "sm_max_mhz": max(r[2] for r in rows) if rows else None,
                    "power_w_max": max(r[3] for r in rows) if rows else None, "reasons": reasons, "samples": len(rows),
                    "source": "nvml, 1 ms period, inside the timed region"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i] == "Active"})
        pw = [float(r[2]) for r in self.rows if len(r) >= 7 and r[2].replace(".", "").isdigit()]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "reasons": reasons, "samples": len(sm), "source": "nvidia-smi -lms 100"}


def cgroup_cpu_quota():
    """CPUs the container may use according to its cgroup (cpu.max / cfs quota), or None when unlimited."""
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        return None if q == "max" else float(q) / float(p)
    except (OSError, ValueError):
        pass
    try:
        q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        return None if q <= 0 else q / p
    except (OSError, ValueError):
        return None


def host_threads():
    """Threads the CPU arm may use: the affinity mask capped by the cgroup CPU quota, not the machine's core count."""
    try:
        n = max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        n = os.cpu_count() or 1
    quota = cgroup_cpu_quota()
    if quota:
        n = max(1, min(n, int(quota + 0.999)))
    return n


def cpu_arm(arena, descs, query, steps, warmup, max_s=150.0):
    """Times the oracle (port of the reference algorithm; CRC32 of every page verified on every read like
    Page::crc_validation) on the WHOLE workload: all selected series, every step. The page set is opened once
    (series index + persistent worker pool, like the reference's cached TsmReader metadata and live runtime threads);
    a step is one query. Steps are cut short only if the run would exceed max_s seconds (stated in `sample`; None:
    never). Returns (info, result of the last step, seconds per step)."""
    from oracle import pyoracle as orc
    cores = host_threads()
    op = orc.OpenPages(arena, descs, cores)
    times, pts, res = [], 0, None
    t_begin = time.perf_counter()
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        res, pts = op.scan(query, verify_crc=True, return_points=True)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
        if max_s is not None and time.perf_counter() - t_begin + dt > max_s and len(times) >= 2:
            break
    op.close()
    med = float(np.median(times))
    n_sel = len(query.series_ids) if query.series_ids is not None else None
    info = {"value": pts / med, "unit": "points/s", "cores": cores, "kind": "port",
            "host": {"affinity_cpus": len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else None,
                     "cgroup_cpu_quota": cgroup_cpu_quota(), "os_cpu_count": os.cpu_count()},
            "sample": "the whole workload (%s selected series, %d points) every step, %d of %d steps timed, %d threads "
                      "(persistent pool, series index built once), CRC32 verified per page per step" % (
                          "all" if n_sel is None else str(n_sel), pts, len(times), steps, cores),
            "ms_per_step_median": med * 1e3, "ms_per_step_min": min(times) * 1e3, "ms_per_step_max": max(times) * 1e3}
    return info, res, med


def results_match(got, exp):
    """Integers / counts / min / max bit-exact, f64 sums and means within 1e-6 relative (BASELINE tolerance)."""
    ok = got.names == exp.names
    for j, (col, agg) in enumerate(got.names):
        ok &= bool((got.validity[j] == exp.validity[j]).all())
        m = exp.validity[j]
        if agg == "mean" or (agg == "sum" and got.phys[col] == cabi.TSKV_PT_F64):
            a, b = got.values[j][m].view(np.float64), exp.values[j][m].view(np.float64)
            ok &= bool((np.abs(a - b) <= 1e-6 * np.maximum(np.abs(b), 1e-300)).all())
        else:
            ok &= bool((got.values[j][m] == exp.values[j][m]).all())
    return bool(ok)


DUMP_MAX_BYTES = 64 << 20


def result_arrays(res):
    """ScanResult -> {name: array} as a caller reads it: per output column c<id>_<agg> the typed values as float64
    ([n_groups, n_buckets], 0 where invalid) and c<id>_<agg>_valid as float32 0 / 1."""
    out = {}
    for col, agg in res.names:
        v, ok = res.column(col, agg)
        out["c%d_%s" % (col, agg)] = v.astype(np.float64)
        out["c%d_%s_valid" % (col, agg)] = ok.astype(np.float32)
    return out


def decoded_arrays(pages):
    """[(u64 values, validity)] of decode_pages -> {name: array}, like result_arrays. float64 cannot hold a nanosecond
    timestamp exactly, so each 64-bit value is written as its high and low 32-bit halves."""
    out = {}
    for i, (v, ok) in enumerate(pages):
        out["page%d_values_hi" % i] = (v >> np.uint64(32)).astype(np.float64)
        out["page%d_values_lo" % i] = (v & np.uint64(0xFFFFFFFF)).astype(np.float64)
        out["page%d_valid" % i] = ok.astype(np.float32)
    return out


def dump_outputs(out_dir, arrays):
    """Writes every array as out_dir/<name>.npy. Above DUMP_MAX_BYTES in all, each array is cut to the same share of
    its elements at positions drawn by a fixed seed (flattened, in order), so arrays of one shape keep the same
    positions and two runs with the same arguments compare element for element."""
    os.makedirs(out_dir, exist_ok=True)
    total = sum(a.nbytes for a in arrays.values())
    share = min(1.0, (DUMP_MAX_BYTES - 256 * len(arrays)) / max(total, 1))  # 256: room for each .npy header
    for name, a in arrays.items():
        if share < 1.0:
            flat = a.reshape(-1)
            keep = np.sort(np.random.default_rng(0).choice(flat.size, int(flat.size * share), replace=False))
            a = flat[keep]
        np.save(os.path.join(out_dir, name + ".npy"), a)
    print("bench: wrote %d arrays to %s%s" % (len(arrays), out_dir, "" if share == 1.0 else
                                              " (seeded sample: %.4f of the elements)" % share), file=sys.stderr)


def bench_decode_only(args, rank, world):
    """C1: 1 series x 10 000 i64 points (Delta + simple8b), decode only - tskvgpu_decode_pages vs the oracle's
    column decode (the reference's own CPU bench shape). Single GPU."""
    from oracle import pyoracle as orc
    g = datagen.generate(1, n_fields=1, n_points=10_000, value_kind=datagen.I64_WALK, seed=1)
    config = {"workload": "C1: 1 series x 10000 i64 points, delta + simple8b, decode only", "series_total": 1,
              "points_per_series": 10_000, "selected_series": 1, "sharding": "none"}
    n_pts = 10_000 * 2  # the time page and the value page
    cores = 1
    times = []
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        exp = orc.decode_pages(g.arena, g.descs)
        if i >= args.warmup:
            times.append(time.perf_counter() - t0)
    cpu = {"value": n_pts / float(np.median(times)), "unit": "points/s", "cores": cores, "kind": "port",
           "sample": "both pages of the series, every step, 1 thread (a single series is one task in the reference)"}
    if args.impl == "reference":
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, decoded_arrays(exp))
        print(json.dumps({"impl": "reference", "metric": "decoded points/s", "value": cpu["value"], "unit": "points/s",
                          "n_gpus": args.gpus, "steps": len(times), "warmup": args.warmup,
                          "ms_per_step": float(np.median(times)) * 1e3, "higher_is_better": True, "scaling": "strong",
                          "vs_baseline": None, "dtype": "i64", "data": "synthetic", "config": config, "cpu_baseline": cpu,
                          "e2e": {"value": cpu["value"], "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return 0
    from cnosdb_b200.engine import Engine
    eng = Engine(int(os.environ.get("LOCAL_RANK", "0")))
    pages = eng.upload_pages(g.arena, g.descs)
    dev_ms, e2e = [], []
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        got = eng.decode_pages(pages, g.descs)
        dt = time.perf_counter() - t0
        if i >= args.warmup:
            e2e.append(dt)
            dev_ms.append(eng.counters()["elapsed_scan_ms"])
    ok = all((gm == em).all() and (gv[em] == ev[em]).all() for (gv, gm), (ev, em) in zip(got, exp))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, decoded_arrays(got))
    page_bytes = int(g.descs["size"].sum())
    peak = 6584.5
    try:
        peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except (OSError, ValueError, KeyError):
        pass
    ms = float(np.median(dev_ms))
    algo = page_bytes + 8 * n_pts  # decode-only writes the decoded values
    line = {"metric": "decoded points/s", "value": n_pts / (ms / 1e3), "unit": "points/s", "n_gpus": 1,
            "steps": len(dev_ms), "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "i64", "data": "synthetic", "config": config,
            "e2e": {"value": n_pts / float(np.median(e2e)), "unit": "points/s", "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": 8 * n_pts + n_pts // 8, "ms_per_step": float(np.median(e2e)) * 1e3},
            "gpu_launches": len(dev_ms), "roofline": {"bound": "hbm", "kernel": "k_decode_warp", "achieved": algo / (ms / 1e3) / 1e9,
                                                       "peak": peak, "unit": "GB/s", "frac": algo / (ms / 1e3) / 1e9 / peak,
                                                       "traffic": None, "bound_note": "launch-latency-bound: 2 pages"},
            "cpu_baseline": cpu, "parity_sample": "ok" if ok else "MISMATCH"}
    print(json.dumps(line))
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C4", choices=["C1", "C2", "C3", "C4", "C5"])
    ap.add_argument("--series", type=int, default=0, help="total series (default: the workload's BASELINE size)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result of the last timed step as DIR/<name>.npy (float64 / float32, <= 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.workload == "C1":
        return bench_decode_only(args, rank, world) if rank == 0 else 0
    wl = WORKLOADS[args.workload]
    n_series = args.series or wl.default_series
    steps, warmup = args.steps, max(args.warmup, 3 if args.impl == "ours" else 0)
    sel_all = wl.select(n_series)
    config = wl.config(n_series)

    if args.impl == "reference":
        if rank != 0:
            return 0
        n_ref = min(n_series, 1_000_000)  # a C5-sized page set does not fit host memory comfortably: bounded
        g = wl.generate(0, n_ref)
        sel = wl.select(n_ref)
        info, res, step_s = cpu_arm(g.arena, g.descs, wl.query(sel), steps, args.warmup, max_s=None)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, result_arrays(res))
        if n_ref != n_series:
            info["sample"] = "first %d of %d series; " % (n_ref, n_series) + info["sample"]
        line = {"impl": "reference", "metric": METRIC, "value": info["value"], "unit": "points/s",
                "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup, "ms_per_step": step_s * 1e3,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "i64/f64",
                "data": "synthetic", "config": config, "cpu_baseline": info,
                "e2e": {"value": info["value"], "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "note": "oracle port of the reference algorithm (the Rust reference cannot be compiled in this image)"}
        print(json.dumps(line))
        return 0

    import torch
    import torch.distributed as dist
    from cnosdb_b200.engine import Engine
    from cnosdb_b200.parallel import GatherExchange

    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    t_gen = time.perf_counter()
    lo, hi = shard_range(n_series, rank, world)
    g = wl.generate(lo, hi - lo)
    t_gen = time.perf_counter() - t_gen
    eng = Engine(local_rank)
    # the exchange runs inside the library (NCCL through the C ABI); TSKV_BENCH_TORCH_EXCHANGE=1 keeps torch.distributed's
    use_torch_x = os.environ.get("TSKV_BENCH_TORCH_EXCHANGE", "0") == "1"
    if world > 1 and not use_torch_x:
        from cnosdb_b200.parallel import init_engine_comm
        use_torch_x = not init_engine_comm(eng, rank, world)
    stream = torch.cuda.ExternalStream(eng.stream(), device=device)
    pages = eng.upload_pages(g.arena, g.descs, verify_crc=True)
    q = wl.query(sel_all, multi_rank=world > 1)
    scan = eng.prepare(pages, q)
    exchange = GatherExchange(scan, eng, world, use_torch=use_torch_x) if world > 1 else None
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)  # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    def timed_steps(sc, ex, n):
        """n steps of the device-resident pass, each bracketed by CUDA events on the engine stream; L2 flushed before
        every step outside the timed interval. Returns the summed milliseconds."""
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
        with torch.cuda.stream(stream):
            for a, b in ev:
                flush.zero_()
                a.record(stream)
                sc.enqueue()
                if ex is not None:
                    ex.run()
                sc.finalize_device()
                b.record(stream)
        sc.sync()
        return sum(a.elapsed_time(b) for a, b in ev)

    # ---- device-resident throughput (value) ------------------------------------------------------
    timed_steps(scan, exchange, warmup)
    c = eng.counters()
    points_local = c["points_decoded"]
    launches_per_step = c["kernel_launches"] + 1
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    t_region = time.perf_counter()
    dev_ms = timed_steps(scan, exchange, steps)
    barrier()
    clocks = sampler.stop(t_region, time.perf_counter()) if rank == 0 else None
    if args.dump_outputs and rank == 0:  # finalize() re-reads the last step's state; the roofline runs below overwrite it
        dump_outputs(args.dump_outputs, result_arrays(scan.finalize()))
    t = torch.tensor([dev_ms, float(points_local)], dtype=torch.float64, device=device)
    if world > 1:
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        dev_ms, points_total = float(tmax[0]), float(t[1])
    else:
        points_total = float(points_local)
    value = points_total * steps / (dev_ms / 1e3)

    # ---- the same with Page::crc_validation on every read: CRC32 of every selected page re-checked per step -----
    pages_crc = eng.upload_pages(g.arena, g.descs, verify_crc=False, verify_on_read=True)
    scan_crc = eng.prepare(pages_crc, q)
    ex_crc = GatherExchange(scan_crc, eng, world, use_torch=use_torch_x) if world > 1 else None
    timed_steps(scan_crc, ex_crc, 2)
    barrier()
    crc_ms = timed_steps(scan_crc, ex_crc, steps)
    tc = torch.tensor([crc_ms], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(tc, op=dist.ReduceOp.MAX)
    value_crc = points_total * steps / (float(tc[0]) / 1e3)
    scan_crc.close()
    pages_crc.close()

    # ---- roofline of the fused phase (live CUDA events inside the library) -------------------------------
    dom_ms, dom_bytes, fused_ms, scan_ms, dom_bin = [], 0, [], [], 0
    for _ in range(max(3, min(steps, 10))):
        with torch.cuda.stream(stream):
            flush.zero_()
        scan.run()
        c = eng.counters()
        dom_ms.append(c["dominant_kernel_ms"])
        fused_ms.append(c["elapsed_fused_ms"])
        scan_ms.append(c["elapsed_scan_ms"])
        dom_bytes, dom_bin = c["dominant_kernel_bytes"], c["dominant_kernel_bin"]
    page_bytes = c["page_read_bytes"]
    L = scan.layout
    n_sel = n_series if sel_all is None else len(sel_all)
    algo_bytes = page_bytes + 24 * c["page_read_count"] + 4 * n_sel + 8 * int(L.n_out * L.n_cells)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except (OSError, ValueError):
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    # `achieved` = the algorithmic bytes of one step / the CUDA-event time from the fork to the join of the fused
    # kernels (one instantiation of k_scan_aggregate<TK,VK,SEL> per decode-kind bin, launched on concurrent streams).
    fused_s = float(np.mean(fused_ms)) * 1e-3
    traffic = None
    if world == 1 and args.workload == "C4" and n_series == wl.default_series:
        try:  # DRAM bytes of the same launches from the committed `ncu --set full` capture (profiles/)
            traffic = json.load(open(os.path.join(ROOT, "profiles", "r02c_scan_ncu_summary.json")))["step_dram_traffic_bytes"]
        except (OSError, ValueError, KeyError):
            pass
    roofline = {"bound": "hbm", "kernel": "k_scan_aggregate<TK,VK,SEL> (fused decode+filter+bucket-reduce), one launch "
                                          "per decode-kind bin on concurrent streams; fork-to-join time",
                "achieved": algo_bytes / fused_s / 1e9, "peak": peak, "unit": "GB/s",
                "frac": algo_bytes / fused_s / 1e9 / peak,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s (of fallback)",
                "traffic": traffic, "bytes_per_launch": int(algo_bytes), "ms_per_launch": fused_s * 1e3,
                "decoded_equivalent_frac": 16 * points_local / fused_s / 1e9 / peak,
                "slowest_bin": {"kernel": "fused scan kernel of bin <%s>" % BIN_NAMES[int(dom_bin)],
                                "ms": float(np.mean(dom_ms)), "page_bytes": int(dom_bytes),
                                "gbs": dom_bytes / max(float(np.mean(dom_ms)), 1e-9) / 1e6},
                "step_ms": float(np.mean(scan_ms)),
                "bound_note": "integer-pipe-bound lane-per-page-part decode (see DESIGN.md section 5 and profiles/)"}

    # ---- end to end: pages in host memory, PCIe gather inside the timed region ---------------------
    # Page CRC32s are re-checked on the device after every transfer (what the reference does on every page read, and
    # what the CPU arm does); TSKV_BENCH_E2E_CRC=0 measures the transfer + scan alone.
    e2e_crc = os.environ.get("TSKV_BENCH_E2E_CRC", "1") != "0"
    hp = eng.upload_pages(g.arena, g.descs, verify_crc=e2e_crc, host_resident=True)

    def e2e_step():
        s = eng.prepare(hp, q)
        s.enqueue()
        if world > 1:
            GatherExchange(s, eng, world, use_torch=use_torch_x).run()
        res = s.finalize()
        s.sync()
        cc = eng.counters()
        s.close()
        return res, cc

    for _ in range(max(1, warmup // 2)):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        res, cc = e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_s = float(te[0])
    e2e = {"value": points_total * steps / e2e_s, "unit": "points/s",
           "crc_verified": "device, every step" if e2e_crc else "off",
           "h2d_bytes_per_step": int(cc["page_read_bytes"] + cc["h2d_bytes"]),
           "d2h_bytes_per_step": int(L.values_bytes + L.validity_bytes + 12 + 13 * 8),
           "ms_per_step": e2e_s / steps * 1e3,
           "path": "prepare(H2D args) + select + PCIe gather of selected pages + device CRC32 + fused scan + finalize(D2H)"}
    hp.close()

    # ---- CPU baseline + parity ------------------------------------------------------------------------------
    # N = 1: the CPU arm runs the whole workload, so the comparison covers every selected series.
    # N > 1: a sample made of one block of series from EVERY shard is scanned by all ranks and exchanged like the real
    # query; rank 0 rebuilds those blocks' pages, runs the oracle and compares; every rank's merged result must be
    # byte-identical to rank 0's.
    cpu, parity = None, None
    if world == 1:
        if not args.no_cpu_baseline:
            cpu, cpu_res, _ = cpu_arm(g.arena, g.descs, wl.query(sel_all), 2, 1)
            parity = "ok" if results_match(eng.scan_aggregate(pages, wl.query(sel_all)), cpu_res) else "MISMATCH"
    else:
        from oracle import pyoracle as orc
        block = 2048
        blocks = []
        for r in range(world):
            blo, bhi = shard_range(n_series, r, world)
            blocks.append((blo, min(block, bhi - blo)))
        ids = np.concatenate([np.arange(b, b + n, dtype=np.uint32) for b, n in blocks])
        if sel_all is not None:
            ids = np.intersect1d(ids, sel_all).astype(np.uint32)
        qs = wl.query(ids, multi_rank=True)
        s = eng.prepare(pages, qs)
        s.enqueue()
        GatherExchange(s, eng, world, use_torch=use_torch_x).run()
        got = s.finalize()
        s.sync()
        s.close()
        digest = zlib.crc32(got.values.tobytes() + got.validity.tobytes())
        dg = torch.tensor([digest], dtype=torch.int64, device=device)
        all_dg = [torch.zeros_like(dg) for _ in range(world)]
        dist.all_gather(all_dg, dg)
        same = all(int(x) == int(all_dg[0]) for x in all_dg)
        if rank == 0:
            parts = []
            for b, n in blocks:
                gb = wl.generate(b, n)
                parts.append((gb.arena.copy(), gb.descs.copy()))
                gb.close()
            arena_s, descs_s = concat_arenas(parts)
            exp = orc.scan_aggregate(arena_s, descs_s, wl.query(ids), n_threads=host_threads())
            ok = results_match(got, exp)
            parity = ("ok" if ok and same else "MISMATCH") + " (%d series from %d shards, merged result identical on all ranks: %s)" % (
                len(ids), world, same)

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "points/s", "n_gpus": world, "steps": steps,
                "warmup": warmup, "ms_per_step": dev_ms / steps, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "i64/f64", "data": "synthetic", "config": config,
                "run": {"l2_flush_between_steps": True, "pages_resident": "HBM",
                        "exchange": None if world == 1 else ("torch.distributed all_gather + merge kernel" if use_torch_x else "tskvgpu_scan_exchange (ncclAllGather inside the library) + merge kernel"),
                        "encoded_bytes_selected_per_rank": int(page_bytes), "generate_s": round(t_gen, 2)},
                "value_crc_per_step": value_crc, "ms_per_step_crc_per_step": float(tc[0]) / steps,
                "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches_per_step * steps),
                "roofline": roofline, "cpu_baseline": cpu, "parity_sample": parity,
                "points_per_step": points_total}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
