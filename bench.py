#!/usr/bin/env python
"""bench.py -- TFRecord decode GB/s on BASELINE.json's configs[1] workload.

    python bench.py --gpus N --steps K --warmup W            # our arm (one process per GPU under torchrun)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path on the host cores

Workload: configs[1] = 10 M unique synthetic Example records (32 x Int64List[1] + 16 x FloatList[8] + 16 x BytesList[1] of
16 B, entries in schema order), held as a pool of 16 distinct 1 GiB batches of framed TFRecord bytes per GPU, CRC verified,
decoded to Arrow-layout columns.  A "step" is --batches-per-step (64) batch decodes cycling through the pool = four passes
over the 10 M records, so that the default 16 timed steps are about one second of device time.  Prints ONE JSON line (rank 0).

  value  : framed input GB/s with the pool resident in HBM (CUDA events on the decoder's stream around exactly K steps,
           max over ranks), through the pipelined C-ABI call tfr_decode_submit.
  e2e    : the same metric with HOST buffers: every batch is copied from pinned host memory to the device, decoded, and
           all Arrow buffers are copied back to pinned host memory (what a row-based Spark consumer needs), ONE decoder
           handle on ONE thread (tfr_decode_submit + tfr_batch_to_host_async keep H2D / kernels / D2H overlapped).
  roofline: the dominant kernel (decode_tile_kernel: the whole decode in one pass -- reads the framed input once, writes
           every Arrow byte once): algorithmic bytes per launch / its mean launch time (CUDA events recorded by the library
           around every launch in the timed region), against the HBM copy bandwidth this run measures on the same GPU.
  parity_checked: after the timed loop one pool batch is decoded again in the very mode that was timed and compared, bit
           for bit and over all of its records, with the CPU oracle.
  cpu_baseline: the oracle port (C restatement of the reference's per-record algorithm) on the host cores.
  extra  : side metrics, each with its own roofline: configs[2] encode, configs[3] SequenceExample decode, configs[1]
           with ragged bytes columns, ByteArray records.

  --dump-outputs DIR: after the timed steps, the columns the last decode of the last timed step returned are written to
           DIR as float .npy files (see dump_outputs), so that two builds can be compared output for output: with the same
           arguments the inputs are the same seeded records in every run.

The synthetic columns are seeded numpy data; our arm frames them with the product's GPU encoder (proved byte-identical
to the reference writer by tests/test_gpu_encode.py and tests/test_gpu_scale.py), the CPU arm with the oracle's writer.
Nothing under oracle/ is executed outside the parity check, the cpu_baseline leg and the --impl reference arm.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
import zlib
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "TFRecord decode GB/s (1 KB Example, 64 mixed features) at 1/2/4/8 B200"
UNIT = "GB/s"
REC_BYTES = 1728          # mean framed record size of the configs[1] schema (measured; printed in the config)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=16)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch-mib", type=int, default=1024, help="framed bytes per batch (approx.)")
    ap.add_argument("--pool", type=int, default=16, help="distinct batches resident in HBM (16 x 1 GiB = the 10 M records of configs[1])")
    ap.add_argument("--batches-per-step", type=int, default=64, help="batch decodes per step (cycling through the pool)")
    ap.add_argument("--e2e-batches-per-step", type=int, default=4, help="batch decodes per step of the host-buffer (e2e) measurement")
    ap.add_argument("--cpu-sample-mib", type=int, default=48, help="framed bytes each host thread decodes per pass (at most batch / threads)")
    ap.add_argument("--cfg5-passes", type=int, default=4, help="passes over the 200 GB logical corpus in the configs[4] side measurement (0: skip)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed decode returned to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.dump_outputs is not None and (args.impl != "ours" or args.steps < 1):
        ap.error("--dump-outputs writes the last timed step of the GPU arm: it needs --impl ours and --steps >= 1")
    return args


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


# ---------------------------------------------------------------------------------------------
# corpus: configs[1] records.  The columns are seeded numpy data; our arm frames them with the product's own GPU encoder
# (tests prove its bytes identical to the reference writer's), the CPU arm with the oracle's writer: the oracle is executed
# only by the parity check and the CPU legs of this file.
# ---------------------------------------------------------------------------------------------
def cfg2_schema():
    from spark_tfrecord_b200.sqltypes import ArrayType, BinaryType, FloatType, LongType, StructField, StructType
    fields = [StructField(f"i{i:02d}", LongType()) for i in range(32)]
    fields += [StructField(f"f{i:02d}", ArrayType(FloatType())) for i in range(16)]
    fields += [StructField(f"b{i:02d}", BinaryType()) for i in range(16)]
    return StructType(fields)


def cfg2_schema_and_columns(n: int, seed: int, ragged_bytes: bool = False):
    """32 x Int64List[1], 16 x FloatList[8], 16 x BytesList[1] (16 B), entries in schema order (same generator and seeds as
    the parity tests' corpus).  ragged_bytes: the bytes columns get 0..40 bytes per row instead of 16."""
    from spark_tfrecord_b200._cabi import HostColumn
    from spark_tfrecord_b200.sqltypes import TFR_T_BINARY, TFR_T_FLOAT32, TFR_T_INT64
    rng = np.random.Generator(np.random.PCG64(seed))
    valid = np.full((n + 7) // 8, 0xFF, dtype=np.uint8)
    if n % 8 and len(valid):
        valid[-1] = (1 << (n % 8)) - 1
    cols = []
    for i in range(32):
        v = rng.integers(0, 2**21, n, dtype=np.int64)
        if i % 8 == 7:          # quarter each of [0,127], [128,2^31), [-2^31,0), full int64
            sel = rng.integers(0, 4, n)
            a = rng.integers(0, 128, n, dtype=np.int64)
            b = rng.integers(128, 2**31, n, dtype=np.int64)
            c = rng.integers(-2**31, 0, n, dtype=np.int64)
            d = rng.integers(-2**63, 2**63 - 1, n, dtype=np.int64, endpoint=True)
            v = np.choose(sel, [a, b, c, d])
        cols.append(HostColumn(TFR_T_INT64, 0, n, valid, [], v))
    for i in range(16):
        vals = rng.standard_normal(n * 8, dtype=np.float32)
        cols.append(HostColumn(TFR_T_FLOAT32, 1, n, valid, [(np.arange(n + 1, dtype=np.int64) * 8).astype(np.int32)], vals))
    for i in range(16):
        if ragged_bytes:
            lens = rng.integers(0, 41, n)
            offs = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
            data = rng.integers(0, 256, int(offs[-1]), dtype=np.uint8)
        else:
            offs = (np.arange(n + 1, dtype=np.int64) * 16).astype(np.int32)
            data = rng.integers(0, 256, n * 16, dtype=np.uint8)
        cols.append(HostColumn(TFR_T_BINARY, 0, n, valid, [offs], data))
    return cfg2_schema(), cols


def records_per_batch(batch_mib: int) -> int:
    return max(1, (batch_mib << 20) // REC_BYTES)


def make_host_batches(batch_mib: int, count: int, seed: int):
    """framed by the oracle's writer (CPU arm)"""
    from oracle import oracle
    n = records_per_batch(batch_mib)
    out = []
    schema = None
    for i in range(count):
        schema, cols = cfg2_schema_and_columns(n, seed=seed + 1000 * i)
        data, rc, _ = oracle.encode(cols, schema)
        assert rc == 0
        out.append(np.frombuffer(data, dtype=np.uint8))
    return schema, n, out


def make_device_pool(batch_mib: int, pool: int, seed: int, device: int, keep_host: int):
    """`pool` distinct batches framed by the product's encoder on `device`, kept there as torch uint8 tensors; the first
    `keep_host` are also returned as host arrays (e2e staging, CPU baseline, parity check)"""
    import torch
    from spark_tfrecord_b200 import _native
    n = records_per_batch(batch_mib)
    schema = cfg2_schema()
    enc = _native.Encoder(schema, 0, device)
    dev, host = [], []
    with ThreadPoolExecutor(max_workers=min(4, pool)) as ex:       # numpy's generators release the GIL while they fill
        futs = [ex.submit(cfg2_schema_and_columns, n, seed + 1000 * i) for i in range(pool)]
        for i, f in enumerate(futs):
            _, cols = f.result()
            data = np.frombuffer(enc.encode(cols), dtype=np.uint8)
            dev.append(torch.from_numpy(data.copy()).cuda(device))
            if i < keep_host:
                host.append(data)
            del cols
    enc.close()
    return schema, n, dev, host


def host_mem_available():
    """bytes of host memory this process tree may still take: MemAvailable capped by the cgroup limit"""
    avail = None
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable:"):
                avail = int(line.split()[1]) * 1024
    except Exception:
        pass
    try:
        mx = open("/sys/fs/cgroup/memory.max").read().strip()
        if mx != "max":
            cur = int(open("/sys/fs/cgroup/memory.current").read())
            room = int(mx) - cur
            avail = room if avail is None else min(avail, room)
    except Exception:
        pass
    return avail


def host_cores():
    """host threads this process may really use: the affinity mask capped by the cgroup CPU quota"""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(int(txt[0]) / int(txt[1]))))
            else:
                q = int(txt[0])
                per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if q > 0:
                    n = min(n, max(1, q // per))
            break
        except Exception:
            continue
    return n


def bind_to_gpu_numa_node(index: int):
    """Pin this rank (and the pinned buffers it allocates from now on: first touch) to the CPUs next to its GPU.  Returns a
    description for the JSON line; never fails the run."""
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
        h = pynvml.nvmlDeviceGetHandleByIndex(idx)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        near = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1}
        cur = os.sched_getaffinity(0)
        want = near & cur
        if not want:
            return {"bound": False, "why": "GPU-local CPUs are outside this process's cpuset"}
        if want != cur:
            os.sched_setaffinity(0, want)
        node = None
        try:
            for d in sorted(os.listdir("/sys/devices/system/node")):
                if d.startswith("node") and d[4:].isdigit():
                    cpus = set()
                    for part in open(f"/sys/devices/system/node/{d}/cpulist").read().strip().split(","):
                        lo, _, hi = part.partition("-")
                        cpus.update(range(int(lo), int(hi or lo) + 1))
                    if want <= cpus:
                        node = int(d[4:])
                        break
        except Exception:
            pass
        return {"bound": True, "cpus": len(want), "numa_node": node}
    except Exception as e:      # noqa: BLE001
        return {"bound": False, "why": f"{type(e).__name__}: {e}"[:120]}


# ---------------------------------------------------------------------------------------------
# CPU arm: the oracle port on all host cores
# ---------------------------------------------------------------------------------------------
def record_starts(batch: np.ndarray) -> np.ndarray:
    offs = [0]
    pos = 0
    n = len(batch)
    while pos + 16 <= n:
        ln = int(batch[pos:pos + 8].view("<u8")[0])
        if pos + 16 + ln > n:
            break
        pos += 16 + ln
        offs.append(pos)
    return np.array(offs, dtype=np.int64)


def record_aligned_slices(batch: np.ndarray, n_slices: int, slice_bytes: int, offs=None):
    """[(start, end)] of disjoint record-aligned windows spread evenly over the batch"""
    offs = record_starts(batch) if offs is None else offs
    n = int(offs[-1])
    slice_bytes = min(slice_bytes, n // max(1, n_slices))
    out = []
    for i in range(n_slices):
        lo = i * n // n_slices
        si = int(np.searchsorted(offs, lo))
        s = int(offs[min(si, len(offs) - 1)])
        ei = int(np.searchsorted(offs, min(n, s + slice_bytes), side="right")) - 1
        e = int(offs[max(ei, si)])
        if e > s:
            out.append((s, e))
    return out


def cpu_pass(schema, batch, slices):
    """one thread per slice decodes it with the oracle; returns (bytes, seconds)"""
    from oracle import oracle
    oracle.lib()
    errs = []

    def work(i):
        s, e = slices[i]
        r = oracle.decode(batch[s:e], schema, copy_columns=False)
        if r.info["error_code"] != 0:
            errs.append(r.info)

    ths = [threading.Thread(target=work, args=(i,)) for i in range(len(slices))]
    t0 = time.perf_counter()
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    dt = time.perf_counter() - t0
    assert not errs, errs
    return sum(e - s for s, e in slices), dt


def workload_config(args, n_records, batch_bytes, extra=None):
    c = {"workload": "configs[1]: Example decode, 32xInt64List[1] + 16xFloatList[8] + 16xBytesList[1](16 B), CRC verified, -> Arrow columns",
         "batch_mib": args.batch_mib, "records_per_batch": n_records, "framed_bytes_per_batch": batch_bytes,
         "mean_framed_record_bytes": round(batch_bytes / max(1, n_records), 1),
         "pool_batches": args.pool, "unique_records": n_records * args.pool,
         "batches_per_step": args.batches_per_step, "records_per_step": n_records * args.batches_per_step,
         "framed_bytes_per_step": batch_bytes * args.batches_per_step,
         "l2": "every batch (1 GiB) is 8x the 126 MB L2 and consecutive decodes take different batches of a 16 GiB pool"}
    if extra:
        c.update(extra)
    return c


def run_reference(args):
    rank, world, local = dist_env()
    if rank != 0:
        return
    cores = host_cores()
    schema, n, batches = make_host_batches(args.batch_mib, 1, seed=2024)
    batch = batches[0]
    slices = record_aligned_slices(batch, cores, args.cpu_sample_mib << 20)
    per_pass = sum(e - s for s, e in slices)
    for _ in range(args.warmup):
        cpu_pass(schema, batch, slices)
    tot_b, tot_t = 0, 0.0
    for _ in range(args.steps):
        b, dt = cpu_pass(schema, batch, slices)
        tot_b += b
        tot_t += dt
    v = tot_b / tot_t / 1e9
    line = {
        "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * tot_t / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic", "impl": "reference",
        "config": workload_config(args, n, int(len(batch))),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"each step = {cores} threads x one disjoint record-aligned slice ({per_pass >> 20} MiB in total) of one configs[1] batch "
                                   "of the same size as the GPU arm's; oracle/tfr_oracle.c, the C port of the reference path (the JVM reference cannot run "
                                   "here: no JDK)"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock + throttle reasons sampled with NVML DURING the timed regions (resident + e2e);
    falls back to `nvidia-smi -lms` when pynvml is unavailable."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.index = index
        self.sm, self.reasons, self.max = [], set(), None
        self._stop = threading.Event()
        self.th = None
        self.mode = None
        self.period = float(os.environ.get("TFR_CLOCK_PERIOD_S", "0.02"))

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            # CUDA_VISIBLE_DEVICES may remap indices; the box exposes GPUs in order
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.index]) if vis and vis.split(",")[self.index].isdigit() else self.index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nv = pynvml
            self.mode = "nvml"
            self.th = threading.Thread(target=self._poll, daemon=True)
            self.th.start()
        except Exception:
            self.mode = "smi"
            try:
                q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
                self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "50"],
                                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
                self.lines = []
                self.th = threading.Thread(target=lambda: [self.lines.append(l.strip()) for l in self.proc.stdout], daemon=True)
                self.th.start()
            except Exception:
                self.mode = None

    def _poll(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        if self.mode == "nvml":
            self._stop.set()
            self.th.join(timeout=1)
            return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max, "reasons": sorted(self.reasons),
                    "samples": len(self.sm), "source": f"nvml, {int(self.period * 1000)} ms period, resident + e2e timed regions"}
        if self.mode == "smi":
            time.sleep(0.1)
            self.proc.terminate()
            sm, mx, reasons = [], None, set()
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            for ln in self.lines:
                p = [x.strip() for x in ln.split(",")]
                if len(p) < 6:
                    continue
                try:
                    sm.append(float(p[0])); mx = float(p[1])
                except ValueError:
                    continue
                for nm, v in zip(names, p[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi -lms 50"}
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock sampling unavailable"], "samples": 0}


# ---------------------------------------------------------------------------------------------
# parity inside the bench: the timed mode, one whole batch, bit for bit against the oracle
# ---------------------------------------------------------------------------------------------
def parity_check(dec, schema, d_batch, h_batch, threads):
    """decode d_batch exactly as the timed loop does (pipelined submit in steady state) and compare every record with
    the oracle's decode of the same bytes (threads over record-aligned slices)"""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle import oracle
    from util import assert_columns_equal, slice_columns
    s0 = dec.stats()
    b = dec.submit(d_batch)
    got = b.to_host()
    info = dict(b.info)
    b.release()
    s1 = dec.stats()
    speculative = s1["speculative_submits"] == s0["speculative_submits"] + 1 and s1["speculative_redone"] == s0["speculative_redone"]
    offs = record_starts(h_batch)
    n = len(offs) - 1
    assert info["error_code"] == 0 and info["n_rows"] == n, info
    cuts = [int(round(i * n / threads)) for i in range(threads + 1)]
    errs = []

    def work(i):
        r0, r1 = cuts[i], cuts[i + 1]
        if r1 <= r0:
            return
        try:
            want = oracle.decode(h_batch[offs[r0]:offs[r1]], schema)
            assert want.info["error_code"] == 0 and want.n_rows == r1 - r0
            assert_columns_equal(slice_columns(got, r0, r1), want.columns, schema.names, f"bench parity rows [{r0},{r1})")
        except BaseException as e:      # noqa: BLE001
            errs.append(e)

    ths = [threading.Thread(target=work, args=(i,)) for i in range(threads)]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    if errs:
        raise errs[0]
    return {"records": n, "columns": len(got), "bit_exact": True,
            "mode": "steady state: uniform-shape speculation, rows counted on the device, pipelined submit" if speculative else "synchronising path",
            "against": "oracle/tfr_oracle.c over the whole batch (record-aligned slices, one host thread each)"}


# ---------------------------------------------------------------------------------------------
# --dump-outputs: what the timed path returned, as float .npy files
# ---------------------------------------------------------------------------------------------
DUMP_ROWS = 8192            # rows of the seeded sample written value by value
DUMP_SEED = 7
DUMP_LIMIT = 64 << 20       # bytes of all files together


def _exact_float(a: np.ndarray) -> np.ndarray:
    """`a` as float32 / float64 without rounding: floats stay, bytes and int32 widen exactly, and an int64 becomes two
    float64 columns (signed high word, unsigned low word)"""
    if a.dtype in (np.float32, np.float64):
        return a
    if a.dtype == np.uint8:
        return a.astype(np.float32)
    if a.dtype == np.int32:
        return a.astype(np.float64)
    if a.dtype == np.int64:
        return np.stack([(a >> 32).astype(np.float64), (a & 0xFFFFFFFF).astype(np.float64)], axis=1)
    raise TypeError(f"no exact float form for {a.dtype}")


def dump_outputs(out_dir, names, cols):
    """Writes the host copy of a decoded batch to out_dir and returns the bytes written:
      digest.npy        per column: n_rows, null_count, CRC-32 of its validity bits, of its offsets and of its values (over
                        every row), number of values
      rows.npy          a fixed, seeded sample of row indices
      valid.npy         validity (0/1) of the sampled rows, one row per column
      <name>.npy        the values of the sampled rows, in row order (int64 as [high word, low word] pairs)
      <name>.lengths.npy  for list and bytes columns: the number of values of each sampled row"""
    os.makedirs(out_dir, exist_ok=True)
    n = cols[0].n_rows if cols else 0
    rows = np.sort(np.random.default_rng(DUMP_SEED).choice(n, size=min(n, DUMP_ROWS), replace=False))
    arrays = {"rows": rows.astype(np.float64)}
    digest, valid = [], []
    for name, c in zip(names, cols):
        bits = np.ones(n, np.uint8) if c.validity is None else np.unpackbits(c.validity, bitorder="little")[:n]
        digest.append([c.n_rows, c.null_count, zlib.crc32(np.packbits(bits, bitorder="little").tobytes()),
                       zlib.crc32(b"".join(o.tobytes() for o in c.offsets)), zlib.crc32(c.values.tobytes()), len(c.values)])
        valid.append(bits[rows].astype(np.float32))
        lo, hi = rows, rows + 1
        for o in c.offsets:                 # a row's children are one contiguous range at every level
            lo, hi = o[lo].astype(np.int64), o[hi].astype(np.int64)
        lens = hi - lo
        if c.offsets:
            arrays[f"{name}.lengths"] = lens.astype(np.float64)
        idx = np.repeat(lo - (np.cumsum(lens) - lens), lens) + np.arange(int(lens.sum()))
        arrays[name] = _exact_float(c.values[idx])
    arrays["valid"] = np.array(valid, dtype=np.float32)
    arrays["digest"] = np.array(digest, dtype=np.float64)
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_LIMIT, f"--dump-outputs would write {total} bytes (limit {DUMP_LIMIT})"
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), a)
    return total


def hbm_copy_gbs(torch, dev, reps=10):
    """HBM bandwidth as a device-to-device copy reaches it (bytes read + bytes written): 1 Gi bf16 elements, best of `reps`"""
    a = torch.empty(1 << 30, dtype=torch.bfloat16, device=dev)
    b = torch.empty_like(a)
    b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    best = float("inf")
    for _ in range(reps):
        e0.record()
        b.copy_(a)
        e1.record()
        e1.synchronize()
        best = min(best, e0.elapsed_time(e1))
    return 2 * a.nbytes / (best * 1e-3) / 1e9


# ---------------------------------------------------------------------------------------------
# side metrics (rank 0, N = 1): each a short resident loop with its own roofline
# ---------------------------------------------------------------------------------------------
def _roof(alg_bytes, ms, peak):
    a = alg_bytes / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
    return {"bound": "hbm", "achieved": a, "peak": peak, "unit": "GB/s", "frac": a / peak}


def _time_decoder(torch, dec, d_batches, reps):
    stream = torch.cuda.ExternalStream(dec.stream())
    for i in range(3):
        b, _ = dec.decode(d_batches[i % len(d_batches)])
        assert b.info["error_code"] == 0, b.info
        out_bytes, n_rows = b.info["out_bytes"], b.info["n_rows"]
        b.release()
    for i in range(6):                                   # untimed: the pipelined path with three batches in flight (its pools fill up here)
        dec.submit(d_batches[i % len(d_batches)]).release()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    tot = 0
    for i in range(reps):
        b = dec.submit(d_batches[i % len(d_batches)])
        b.release()
        tot += d_batches[i % len(d_batches)].numel()
    e1.record(stream)
    torch.cuda.synchronize()
    return tot, e0.elapsed_time(e1), out_bytes, n_rows


def run_extras(torch, dev, peak):
    from spark_tfrecord_b200 import _native
    from spark_tfrecord_b200._cabi import HostColumn, tfr_column
    from spark_tfrecord_b200.sqltypes import (ArrayType, FloatType, LongType, StructField, StructType, TFR_T_FLOAT32, TFR_T_INT64,
                                              byte_array_schema, TFR_T_BINARY)
    out = {}
    n = records_per_batch(256)

    # ---- configs[2]: encode, columns resident in HBM -> framed bytes ----
    schema, cols = cfg2_schema_and_columns(n, seed=4242)
    keep, dcols = [], []
    for c in cols:
        t = tfr_column()
        hc = c.to_ctypes()
        for f, _ in tfr_column._fields_:
            setattr(t, f, getattr(hc, f))
        v = torch.from_numpy(c.validity).cuda(dev); keep.append(v); t.validity = v.data_ptr()
        for l, o in enumerate(c.offsets):
            ot = torch.from_numpy(o).cuda(dev); keep.append(ot); t.offsets[l] = ot.data_ptr()
        vt = torch.from_numpy(c.values.view(np.uint8)).cuda(dev); keep.append(vt); t.values = vt.data_ptr()
        dcols.append(t)
    enc = _native.Encoder(schema, 0, dev)
    stream = torch.cuda.ExternalStream(enc.stream())
    for _ in range(3):
        _, nb = enc.encode_columns(dcols, True)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 12
    e0.record(stream)
    for _ in range(reps):
        enc.encode_columns(dcols, True)
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    in_bytes = sum(c.nbytes() for c in cols)
    framed = np.frombuffer(enc.result_host(), dtype=np.uint8)
    out["cfg3_encode"] = {"workload": f"configs[2]: {n} rows x 64 columns resident in HBM -> framed TFRecord bytes (CRC framed, byte-identical to the reference writer)",
                          "value": nb / (ms * 1e-3) / 1e9, "unit": "GB/s of framed output", "ms_per_batch": ms,
                          "roofline": dict(_roof(in_bytes + nb, ms, peak), algorithmic_bytes=in_bytes + nb,
                                           note="whole encode call (size pass + scan + emit + the call's host synchronisation) against columns read once + framed bytes written once")}
    enc.close()
    del keep, dcols

    # ---- configs[1] with ragged bytes columns (0..40 B): one pass, look-back across tiles ----
    schema_r, cols_r = cfg2_schema_and_columns(n, seed=777, ragged_bytes=True)
    enc = _native.Encoder(schema_r, 0, dev)
    d_r = [torch.from_numpy(np.frombuffer(enc.encode(cols_r), dtype=np.uint8).copy()).cuda(dev)]
    enc.close()
    dec = _native.Decoder(schema_r, 0, dev)
    tot, ms, ob, nr = _time_decoder(torch, dec, d_r, 24)
    out["cfg2_ragged_bytes"] = {"workload": f"configs[1] with BytesList values of 0..40 bytes ({nr} records per batch): variable-width columns are not uniform",
                                "value": tot / ms / 1e6, "unit": UNIT, "ms_per_batch": ms / 24, "stats": dec.stats(),
                                "roofline": dict(_roof(d_r[0].numel() + ob, ms / 24, peak), algorithmic_bytes=d_r[0].numel() + ob, note="whole step (frame index + the single-pass tile kernel: tile-local prefix sums + decoupled look-back across tiles)")}
    dec.close()

    # ---- configs[3]: SequenceExample, FeatureList of FloatList (ragged, mean 64 steps) ----
    rng = np.random.Generator(np.random.PCG64(77))
    ns = 120_000
    steps = rng.poisson(64, ns).astype(np.int64)
    o0 = np.concatenate([[0], np.cumsum(steps)]).astype(np.int32)
    inner = rng.integers(1, 9, int(o0[-1])).astype(np.int64)
    o1 = np.concatenate([[0], np.cumsum(inner)]).astype(np.int32)
    valid = np.full((ns + 7) // 8, 0xFF, dtype=np.uint8)
    sch4 = StructType([StructField("id", LongType()), StructField("seq", ArrayType(ArrayType(FloatType())))])
    cols4 = [HostColumn(TFR_T_INT64, 0, ns, valid, [], rng.integers(0, 2**40, ns, dtype=np.int64)),
             HostColumn(TFR_T_FLOAT32, 2, ns, valid, [o0, o1], rng.standard_normal(int(o1[-1]), dtype=np.float32))]
    enc = _native.Encoder(sch4, 1, dev)
    d_4 = [torch.from_numpy(np.frombuffer(enc.encode(cols4), dtype=np.uint8).copy()).cuda(dev)]
    enc.close()
    dec = _native.Decoder(sch4, 1, dev)
    tot, ms, ob, nr = _time_decoder(torch, dec, d_4, 24)
    out["cfg4_sequence_example"] = {"workload": f"configs[3]: {nr} SequenceExample records, FeatureList of FloatList[1..8], Poisson(64) steps -> list<list<float32>>",
                                    "value": tot / ms / 1e6, "unit": UNIT, "ms_per_batch": ms / 24,
                                    "roofline": dict(_roof(d_4[0].numel() + ob, ms / 24, peak), algorithmic_bytes=d_4[0].numel() + ob, note="whole step")}
    dec.close()

    # ---- ByteArray records (1 KiB payloads): framing + CRC only ----
    nb_rec = 500_000
    payload = rng.integers(0, 256, nb_rec * 1024, dtype=np.uint8)
    schb = byte_array_schema()
    colsb = [HostColumn(TFR_T_BINARY, 0, nb_rec, np.full((nb_rec + 7) // 8, 0xFF, np.uint8), [(np.arange(nb_rec + 1, dtype=np.int64) * 1024).astype(np.int32)], payload)]
    enc = _native.Encoder(schb, 2, dev)
    d_b = [torch.from_numpy(np.frombuffer(enc.encode(colsb), dtype=np.uint8).copy()).cuda(dev)]
    enc.close()
    dec = _native.Decoder(schb, 2, dev)
    tot, ms, ob, nr = _time_decoder(torch, dec, d_b, 24)
    out["byte_array"] = {"workload": f"recordType=ByteArray: {nr} records of 1 KiB, CRC verified -> one binary column (single-pass decode_bytes_kernel, pipelined submit)",
                         "value": tot / ms / 1e6, "unit": UNIT, "ms_per_batch": ms / 24,
                         "roofline": dict(_roof(d_b[0].numel() + ob, ms / 24, peak), algorithmic_bytes=d_b[0].numel() + ob, note="whole step")}
    dec.close()
    # ---- the same rows the other way: ByteArray column resident in HBM -> framed records (encode_bytes_kernel) ----
    try:
        c = colsb[0]
        t = tfr_column()
        hcb = c.to_ctypes()
        for f, _ in tfr_column._fields_:
            setattr(t, f, getattr(hcb, f))
        keepb = [torch.from_numpy(c.validity).cuda(dev), torch.from_numpy(c.offsets[0]).cuda(dev), torch.from_numpy(c.values).cuda(dev)]
        t.validity, t.values = keepb[0].data_ptr(), keepb[2].data_ptr()
        t.offsets[0] = keepb[1].data_ptr()
        enc = _native.Encoder(schb, 2, dev)
        stream = torch.cuda.ExternalStream(enc.stream())
        for _ in range(3):
            _, nbb = enc.encode_columns([t], True)
        torch.cuda.synchronize()
        same = nbb == d_b[0].numel() and bool(torch.equal(torch.frombuffer(bytearray(enc.result_host()), dtype=torch.uint8), d_b[0].cpu()))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(12):
            enc.encode_columns([t], True)
        e1.record(stream)
        torch.cuda.synchronize()
        msb = e0.elapsed_time(e1) / 12
        inb = int(c.values.nbytes + c.offsets[0].nbytes)
        out["byte_array_encode"] = {"workload": f"recordType=ByteArray: {nb_rec} rows of 1 KiB resident in HBM -> framed records (single-pass encode_bytes_kernel, whole tfr_encode call)",
                                    "value": nbb / (msb * 1e-3) / 1e9, "unit": "GB/s of framed output", "ms_per_batch": msb, "bytes_identical_to_the_first_encode": same,
                                    "roofline": dict(_roof(inb + nbb, msb, peak), algorithmic_bytes=inb + nbb, note="whole call incl. its host synchronisations")}
        enc.close()
        del keepb
    except Exception as e:      # noqa: BLE001  (a side metric must not take the headline down)
        out["byte_array_encode"] = {"error": repr(e)}
    return out


# ---------------------------------------------------------------------------------------------
# configs[4]: file-sharded decode of a 200 GB logical corpus, strong scaling over the ranks
# ---------------------------------------------------------------------------------------------
CFG5_FILES = 64
CFG5_BLOCK = 768 << 20          # block size of the streaming reader: does not divide a file, so blocks end inside records


def cfg5_file_sizes(pool_batches: int):
    """64 files, sizes log-uniform in [0.5, 8] GiB rounded to whole pool batches (a file = consecutive whole 1 GiB batches of
    this rank's pool, starting at batch (file index mod pool)): about 200 GB in total"""
    rng = np.random.Generator(np.random.PCG64(5))
    gib = np.exp(rng.uniform(np.log(0.5), np.log(8.0), CFG5_FILES))
    return [int(min(8, max(1, round(x)))) for x in gib]


def run_cfg5(torch, dec, d_batches, batch_bytes, rank, world, passes):
    """Every rank takes the files shard_lpt assigns it (the reference's unit is the unsplittable file, M/DefaultSource.scala:26-29)
    and streams each through tfr_decode_submit in blocks of at most 768 MiB: a block that ends inside a record is submitted as
    non-final, tfr_batch_consumed says where the next block starts as soon as the block's frame index has run (the carry-over of
    a streaming reader; the bytes are already in HBM, so the carry is a pointer, and blocks start at any alignment), and the next
    block is submitted before this one's rows are waited for.  Returns (bytes, device ms, files, blocks)."""
    from spark_tfrecord_b200.sharding import shard_lpt
    sizes = cfg5_file_sizes(len(d_batches))
    nominal = [n * (1 << 30) for n in sizes]
    mine = shard_lpt(nominal, world)[rank]
    stream = torch.cuda.ExternalStream(dec.stream())
    P = len(d_batches)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tot, blocks = 0, 0
    prev = None
    e0.record(stream)
    for _ in range(passes):
        for f in mine:
            for k in range(sizes[f]):                       # the file's batches; a record never straddles two of them
                t = d_batches[(f + k) % P]
                nb = batch_bytes[(f + k) % P]
                pos = 0
                while pos < nb:
                    take = min(CFG5_BLOCK, nb - pos)
                    final_block = pos + take == nb
                    b = dec.submit((t.data_ptr() + pos, take, 1), is_final=final_block and k == sizes[f] - 1)
                    used = b.consumed()                       # where the next block starts: known after the frame index, before the rows
                    assert used > 0 and (used == take or not final_block)
                    if prev is not None:                      # the block before this one: its rows are checked while this one decodes
                        info = prev[0].info
                        assert info["error_code"] == 0 and info["consumed_bytes"] == prev[1], info
                        prev[0].release()
                    prev = (b, used)
                    pos += used
                    tot += used
                    blocks += 1
    if prev is not None:
        info = prev[0].info
        assert info["error_code"] == 0 and info["consumed_bytes"] == prev[1], info
        prev[0].release()
    e1.record(stream)
    torch.cuda.synchronize()
    return tot, e0.elapsed_time(e1), len(mine), blocks, sizes


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------
def run_ours(args):
    rank, world, local = dist_env()
    numa = bind_to_gpu_numa_node(local)       # before CUDA and any pinned allocation
    import torch
    from spark_tfrecord_b200 import _native
    _native.lib()      # fails loudly when libtfrgpu.so is missing
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; there is no CPU fallback for the product path")
    torch.cuda.set_device(local)
    dev = local
    use_dist = world > 1
    if use_dist:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if use_dist:
            dist.barrier()
        torch.cuda.synchronize()

    # host footprint per rank: 3 host batches + 3 pinned staging slots + 3 pinned Arrow buffers + the generator's columns:
    # about 12x the batch.  Keep the default batch only if 8 ranks of it fit the host (the same decision at every N, so the
    # per-GPU work does not change with the number of ranks)
    reduced = False
    avail = host_mem_available()
    while avail is not None and args.batch_mib > 128 and 8 * 12 * (args.batch_mib << 20) > avail:
        args.batch_mib //= 2
        reduced = True
    schema, n_rec, d_batches, h_batches = make_device_pool(args.batch_mib, args.pool, seed=2024 + 7919 * rank, device=dev, keep_host=3)
    batch_bytes = [int(b.numel()) for b in d_batches]
    P = len(d_batches)

    # ---------------- resident path: the metric ----------------
    dec = _native.Decoder(schema, 0, dev)
    stream = torch.cuda.ExternalStream(dec.stream(), device=dev)
    out_bytes = 0
    for i in range(3):                         # the decoder learns record size and column shapes
        b, used = dec.decode(d_batches[i % P])
        assert used == batch_bytes[i % P] and b.info["error_code"] == 0, b.info
        out_bytes = b.info["out_bytes"]
        b.release()

    def resident_steps(steps, k0=0, keep_last=False):
        """`steps` x --batches-per-step pipelined decodes; keep_last: the last batch is returned unreleased"""
        nb = 0
        k = k0
        b = None
        for _ in range(steps):
            for _ in range(args.batches_per_step):
                if b is not None:
                    b.release()               # the work stays enqueued; the lane is recycled when its kernels are done
                b = dec.submit(d_batches[k % P])
                nb += batch_bytes[k % P]
                k += 1
        if b is not None and not keep_last:
            b.release()
            b = None
        return nb, k, b

    _, k, _ = resident_steps(args.warmup)
    torch.cuda.synchronize()
    stats0 = dec.stats()
    dec.set_profiling(True)
    clocks = ClockSampler(dev)
    barrier()
    clocks.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.perf_counter()
    ev0.record(stream)
    in_bytes, k, last = resident_steps(args.steps, k, keep_last=args.dump_outputs is not None and rank == 0)
    ev1.record(stream)
    barrier()
    t_wall = time.perf_counter() - t_wall0
    ms = ev0.elapsed_time(ev1)
    prof = dec.get_profile()
    dec.set_profiling(False)
    stats1 = dec.stats()
    n_timed = args.steps * args.batches_per_step
    timed_stats = {k2: stats1[k2] - stats0[k2] for k2 in stats1}
    # every timed decode ran in the pipelined single-pass mode and none was flagged (a flagged batch would have been redone)
    assert timed_stats["speculative_submits"] == n_timed and timed_stats["speculative_redone"] == 0, timed_stats

    # ---------------- --dump-outputs: the columns the last timed decode returned ----------------
    dumped = None
    if last is not None:
        cols = last.to_host()
        assert last.info["error_code"] == 0, last.info
        dumped = {"dir": args.dump_outputs, "pool_batch": (k - 1) % P, "rows": int(last.n_rows),
                  "sampled_rows": min(int(last.n_rows), DUMP_ROWS), "bytes": dump_outputs(args.dump_outputs, schema.names, cols)}
        last.release()
        del cols

    # ---------------- parity of the timed mode, whole batch ----------------
    parity = None
    if not args.no_parity and rank == 0:
        parity = parity_check(dec, schema, d_batches[0], h_batches[0], max(1, host_cores()))

    # ---------------- configs[4]: file-sharded strong scaling ----------------
    cfg5 = None
    if args.cfg5_passes > 0 and P >= 8:
        barrier()
        c_bytes, c_ms, c_files, c_blocks, c_sizes = run_cfg5(torch, dec, d_batches, batch_bytes, rank, world, args.cfg5_passes)
        barrier()
        cfg5 = (c_bytes, c_ms, c_files, c_blocks, c_sizes)

    # ---------------- the one collective of this project: schema inference + NCCL reduce (N > 1) ----------------
    infer = None
    if use_dist:
        from spark_tfrecord_b200.sharding import allreduce_schema
        inf = _native.Infer(0, dev)
        nb_inf = min(batch_bytes[0], 64 << 20)
        # a record-aligned prefix: non-final block, the consumed count is where the last whole record ends
        barrier()
        t0 = time.perf_counter()
        used = inf.update_block((d_batches[0].data_ptr(), nb_inf, 1), is_final=False)
        local = inf.result()
        t_scan = time.perf_counter() - t0
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        merged = allreduce_schema(local, dist, f"cuda:{dev}")
        torch.cuda.synchronize()
        t_reduce = time.perf_counter() - t0
        assert len(merged) == 64 and used > 0, (len(merged), used)
        infer = {"names": len(merged), "scan_bytes_per_rank": int(used), "scan_ms": 1e3 * t_scan, "allreduce_ms": 1e3 * t_reduce,
                 "collective": "all_gather_object(names) + 2 x all_reduce(MAX) over NCCL"}
        inf.close()

    # ---------------- end to end: pinned host -> device -> pinned host, one handle, one thread ----------------
    e2e = None
    if not args.no_e2e:
        d2h = [0]

        def e2e_setup():
            d2 = _native.Decoder(schema, 0, dev)
            S = d2.num_staging_slots()
            stages = []
            for s in range(S):
                src = h_batches[s % len(h_batches)]
                st = d2.staging_slot(s, src.nbytes)
                st[: src.nbytes] = src            # the JVM side writes file bytes here; not part of the timed region
                stages.append((st, src.nbytes))
            for i in range(3):
                b, used = d2.decode(stages[0][0], nbytes=stages[0][1])
                b.to_host_raw()
                b.release()
            return d2, stages

        def e2e_batches(d2, stages, count, out):
            S = len(stages)
            inflight = [None] * S
            tot = 0
            for i in range(count):
                s = i % S
                if inflight[s] is not None:                 # the slot's previous batch: its Arrow buffers are on the host now
                    ob = inflight[s]
                    ob.to_host_raw()
                    assert ob.info["error_code"] == 0 and ob.info["consumed_bytes"] == stages[s][1]
                    d2h[0] = ob.info["out_bytes"]
                    ob.release()
                b = d2.submit(stages[s][0], nbytes=stages[s][1])   # H2D from pinned memory + kernels, no host sync
                b.to_host_async()                                  # D2H of every Arrow buffer into pinned memory, behind the kernels
                inflight[s] = b
                tot += stages[s][1]
            for ob in inflight:
                if ob is not None:
                    ob.to_host_raw()
                    assert ob.info["error_code"] == 0
                    ob.release()
            out.append(tot)

        def e2e_run(handles, count):
            """`count` batches over len(handles) decoder handles, one host thread each"""
            outs, ths = [], []
            per = [count // len(handles) + (1 if k < count % len(handles) else 0) for k in range(len(handles))]
            for (d2, stages), c in zip(handles, per):
                ths.append(threading.Thread(target=e2e_batches, args=(d2, stages, c, outs)))
            for t in ths:
                t.start()
            for t in ths:
                t.join()
            return sum(outs)

        variants = {}
        handles = [e2e_setup()]
        for n_handles in (1, 2):
            while len(handles) < n_handles:
                handles.append(e2e_setup())
            e2e_run(handles[:n_handles], max(2 * 3 * n_handles, args.warmup))
            barrier()
            t0 = time.perf_counter()
            nbytes_e2e = e2e_run(handles[:n_handles], args.steps * args.e2e_batches_per_step)
            torch.cuda.synchronize()
            barrier()
            variants[n_handles] = (nbytes_e2e, time.perf_counter() - t0)
        e2e_stats = handles[0][0].stats()
        for d2, _ in handles:
            d2.close()
        e2e = (variants, d2h[0], e2e_stats)

    clk = clocks.stop()

    # ---------------- reduce over ranks ----------------
    if use_dist:
        ev = e2e[0] if e2e else {1: (0, 0.0), 2: (0, 0.0)}
        t = torch.tensor([ms, t_wall, ev[1][1], ev[2][1], cfg5[1] if cfg5 else 0.0], dtype=torch.float64, device=f"cuda:{dev}")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        s = torch.tensor([float(in_bytes), float(ev[1][0]), float(ev[2][0]), float(cfg5[0] if cfg5 else 0), float(cfg5[3] if cfg5 else 0)], dtype=torch.float64, device=f"cuda:{dev}")
        dist.all_reduce(s, op=dist.ReduceOp.SUM)
        ms, t_wall, t_e2e_1, t_e2e_2, cfg5_ms_max = t.tolist()
        tot_in, tot_e2e_1, tot_e2e_2, cfg5_bytes, cfg5_blocks = s.tolist()
    else:
        ev = e2e[0] if e2e else {1: (0, 0.0), 2: (0, 0.0)}
        tot_in = float(in_bytes)
        tot_e2e_1, t_e2e_1, tot_e2e_2, t_e2e_2 = float(ev[1][0]), ev[1][1], float(ev[2][0]), ev[2][1]
        cfg5_ms_max, cfg5_bytes, cfg5_blocks = (cfg5[1], float(cfg5[0]), float(cfg5[3])) if cfg5 else (0.0, 0.0, 0.0)

    if rank != 0:
        if use_dist:
            dist.destroy_process_group()
        return

    value = tot_in / (ms * 1e-3) / 1e9
    # ---------------- roofline of the dominant kernel ----------------
    peak = hbm_copy_gbs(torch, dev)
    peak_src = "measured by this run on the same GPU: device copy of 1 Gi bf16 elements (bytes read + written), best of 10"
    p1_alg = batch_bytes[0] + int(out_bytes)        # framed input read once + Arrow output written once (algorithmic bytes of the whole decode of one batch)
    p1_ms = prof["ms"]["pass1"] / max(1, prof["pass1_launches"])
    achieved = p1_alg / (p1_ms * 1e-3) / 1e9 if p1_ms > 0 else 0.0
    ms_per_batch = ms / n_timed
    stage_ms = {k2: round(v / n_timed, 4) for k2, v in prof["ms"].items()}
    traffic = None
    traffic_src = None
    try:
        with open(os.path.join(ROOT, "profiles", "tile_traffic.json")) as f:
            tj = json.load(f)
        traffic = int(tj["dram_bytes_per_framed_byte"] * batch_bytes[0])
        traffic_src = f"ncu dram__bytes_read+write per framed byte of this kernel ({tj['source']}) x this batch; not re-measured by this run"
    except Exception:
        pass
    roof = {"bound": "hbm", "kernel": "decode_tile_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
            "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
            "algorithmic_bytes_per_launch": p1_alg, "kernel_ms_per_launch": p1_ms, "launches_timed": int(prof["pass1_launches"]),
            "share_of_step": p1_ms / ms_per_batch if ms > 0 else None,
            "note": "launch time measured live with CUDA events while the next batch's frame index runs concurrently on a second stream"}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": workload_config(args, n_rec, batch_bytes[0], extra={
            "arrow_out_bytes_per_batch": int(out_bytes),
            "timing": "CUDA events on the decoder's stream around K steps (value); wall clock around the pipelined host-buffer loop incl. copies (e2e); max over ranks",
            "parallelism": f"file/block sharded, {world} rank(s), no collective on the data path",
            "batch_reduced_for_host_memory": reduced, "numa": numa}),
        "ms_per_batch": ms_per_batch,
        "roofline": roof,
        "step_hbm": {"algorithmic_bytes_per_batch": int(p1_alg), "achieved_GBps": p1_alg / (ms_per_batch * 1e-3) / 1e9,
                     "frac_of_peak": p1_alg / (ms_per_batch * 1e-3) / 1e9 / peak, "stage_ms_per_batch": stage_ms,
                     "note": "stages overlap: the frame index (and the uniform columns' offsets) of batch t+1 run on a second stream under the tile kernel of batch t"},
        "pipeline": dict(timed_stats, host_syncs_per_batch=0),
        "clocks": clk,
        "gpu_launches": int(prof["launches"]),
        "wall_s_timed_region": t_wall,
    }
    if parity:
        line["parity_checked"] = parity
    if dumped:
        line["dumped_outputs"] = dumped
    if infer:
        line["schema_inference_reduce"] = infer
    if cfg5:
        corpus = sum(cfg5[4]) * (1 << 30)
        line["cfg5_file_sharded"] = {
            "workload": f"configs[4]: {CFG5_FILES} files of configs[1] records, sizes log-uniform 0.5-8 GiB ({corpus / 1e9:.0f} GB logical corpus), assigned to the "
                        f"{world} rank(s) by LPT on their sizes (the file is the reference's unsplittable unit), each streamed in blocks of <= 768 MiB with carry-over",
            "value": cfg5_bytes / (cfg5_ms_max * 1e-3) / 1e9, "unit": UNIT, "scaling": "strong", "passes_over_corpus": args.cfg5_passes,
            "framed_bytes_decoded": int(cfg5_bytes), "blocks": int(cfg5_blocks), "device_ms_max_over_ranks": cfg5_ms_max,
            "replay": f"each rank's files replay its {P} resident 1 GiB batches ({P * batch_bytes[0] / 1e9:.0f} GB unique per GPU); the logical corpus is decoded {args.cfg5_passes}x",
            "note": "a block's consumed-bytes count is fetched right after its frame index (tfr_batch_consumed): the next block is cut and submitted while this one "
                    "decodes, its rows are checked one block later; each 1 GiB batch goes as a 768 MiB and a 256 MiB block, smaller launches than the headline loop's"}
    if e2e:
        eb = args.e2e_batches_per_step
        v1 = tot_e2e_1 / t_e2e_1 / 1e9 if t_e2e_1 > 0 else 0.0
        v2 = tot_e2e_2 / t_e2e_2 / 1e9 if t_e2e_2 > 0 else 0.0
        line["e2e"] = {"value": max(v1, v2), "unit": UNIT, "h2d_bytes_per_step": int(batch_bytes[0]) * eb,
                       "d2h_bytes_per_step": int(e2e[1]) * eb, "batches_per_step": eb, "steps": args.steps,
                       "one_handle_one_thread": v1, "two_handles_two_threads": v2,
                       "pipeline": "per decoder handle ONE host thread: tfr_decode_submit (H2D on the copy stream, frame index, tile kernel, no host sync) + "
                                   "tfr_batch_to_host_async (D2H on the copy-out stream), 3 pinned staging slots in, pinned Arrow buffers out; value = the better of one "
                                   "handle / one thread and two handles / two threads (what two Spark tasks sharing a GPU do)",
                       "ceiling": "tools/pcie_probe.py on this pool (profiles/r2_pcie_probe_*.json): plain pinned copies of the same sizes in both directions at once move "
                                  "51.7 + 35.1 GB/s on one GPU, 227 + 154 GB/s on eight",
                       "stats": e2e[2]}
    # ---------------- CPU baseline beside it (rank 0, N=1 only) ----------------
    if not args.no_cpu and world == 1:
        cores = host_cores()
        slices = record_aligned_slices(h_batches[0], cores, args.cpu_sample_mib << 20)
        cpu_pass(schema, h_batches[0], slices)
        tb, tt, passes = 0, 0.0, 0
        while tt < 8.0 and passes < 40:
            bb, dt = cpu_pass(schema, h_batches[0], slices)
            tb += bb
            tt += dt
            passes += 1
        line["cpu_baseline"] = {"value": tb / tt / 1e9, "unit": UNIT, "cores": cores, "kind": "port",
                                "sample": f"{cores} threads x one disjoint record-aligned slice of one batch ({sum(e - s for s, e in slices) >> 20} MiB per pass), {passes} passes, {tt:.1f} s of wall time"}
    if not args.no_extra and world == 1:
        try:
            dec.close()
            dec = None
            del d_batches
            torch.cuda.empty_cache()
            line["extra"] = run_extras(torch, dev, peak)
        except Exception as e:      # noqa: BLE001  (side metrics never fail the headline)
            line["extra"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    print(json.dumps(line))
    if dec is not None:
        dec.close()
    if use_dist:
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
