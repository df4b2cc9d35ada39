#!/usr/bin/env python
"""Benchmark of the field-transform hot path on B200 — BASELINE.json's headline metric.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload (config 3 of BASELINE.json, the one the metric is quoted on): regrid 0.25°
(1440x721 = 1,038,240 points) → N320-shaped (542,080 points) with a 4-point bilinear CSR
matrix, 3120 float32 fields (10 vars x 13 levels x 24 steps).  One *step* = one pass of the
matrix over the 3120-field job.  Synthetic data (no network): seeded random fields, a
locally built bilinear matrix, an N320-shaped reduced Gaussian grid (the real N320 `pl`
table is not available offline — same point count and density).

One JSON line on stdout (rank 0):
    value         fields/s with the job resident in HBM (device-timed, max over ranks)
    e2e           fields/s through the reference-facing plugin call:
                  create_filter_by_name("regrid", matrix=…).forward(FieldList of ordinary numpy
                  fields) + to_numpy() of every output — host staging, H2D, kernels and D2H all
                  inside the timed region
    e2e_pinned_fields  the same plugin call on fields whose numpy arrays live in page-locked memory
                  (device.pinned_empty — what a decoder that feeds these filters allocates): no
                  staging copy
    e2e_cabi      the same bytes through the bare C-ABI pipeline (at_pipeline_regrid) with
                  caller-pinned buffers: the PCIe floor the plugin path is measured against
    pipeline_e2e  config 4 as a FieldList pipeline (regrid | uv_to_ddff | q_to_r | clip |
                  apply_mask, O1280 → N320-shaped, 12 nnz/row), with the reference's five-pass
                  CPU chain timed beside it (N = 1)
    e2e_grib      config 3 as a GRIB FieldList (16-bit simple packing): packed octets over PCIe,
                  decoded on the device (float64 like the reference's to_numpy(), and float32),
                  with the reference's decode + scipy chain timed beside it (N = 1)
    roofline      algorithmic bytes per launch / measured launch time vs the measured HBM peak;
                  `traffic` is read from the committed ncu export under profiles/
    cpu_baseline  the reference's CPU path on the box's host cores (bounded sample; three
                  legs, the fastest reported — benchmarks/cpu_reference.py)
    knn           config 2: N320 targets vs 0.25° sources, k=1 (queries sharded over ranks, the
                  indices exchanged over NVLink)

Multi-GPU: one process per GPU (torchrun).  STRONG scaling: the 3120 fields of the one job
are sharded over the ranks (390-392 per GPU at N = 8), no collective on the math path;
`weak` repeats the round-1 figure (3120 fields on every GPU) as an extra key.

--dump-outputs DIR writes, after the timed steps, a fixed sample of what the last timed step
returned (rank 0's Y [target points x fields], float32): DIR/spmm_fields.npy holds whole fields
[542,080 x 12] and DIR/spmm_points.npy every field at a set of target points [2048 x 3120 at
N = 1], 51.6 MB in all.  Inputs are seeded, so two builds run with the same arguments can be
compared output for output.

--impl reference times the reference's CPU path on the host cores of the box, all of them
whatever OMP_NUM_THREADS says, on the same job at every N: scipy per field on one thread (as
the reference runs), scipy `csr @ X` over one process per core, and the oracle's plain-C
restatement under OpenMP; the fastest is the arm.  Each step is a bounded sample of the job.
"""

from __future__ import annotations

import argparse
import csv
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

REPO = Path(__file__).resolve().parent
for p in (str(REPO), str(REPO / "anemoi-transform_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

N_FIELDS = 3120
WORKLOAD = "regrid 0.25deg (1440x721=1,038,240 pts) -> N320-shaped (542,080 pts), 4-nnz bilinear CSR, 3120 float32 fields"
CPU_SAMPLE_FIELDS = 624  # 1/5 of the job per CPU step
NCU_EXPORT = REPO / "profiles" / "r02_spmm_ncu_raw.csv"  # `ncu --set full … --page raw --csv` of bench.py --value-only


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def bench_config(world: int) -> dict:
    """The `config` object — identical in both arms."""
    return {
        "workload": WORKLOAD,
        "fields_total": N_FIELDS,
        "layout": "point-major [points x fields] float32 in HBM",
        "l2": "inputs larger than L2 (X 12.96 GB + Y 6.77 GB per step over all ranks; >= 2.4 GB per rank at N=8), no flush needed",
        "parallelism": f"the 3120 fields sharded over {world} GPU(s) (strong scaling), no collective on the math path",
    }


def measured_peak_gbs() -> tuple[float, str]:
    f = REPO / "MEASURED_PEAKS.json"
    if f.exists():
        try:
            return float(json.loads(f.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic_bytes(kernel_substring: str = "spmm_f32_kernel"):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the SpMM kernel, from the
    committed `ncu --page raw --csv` export (None when there is no capture)."""
    if not NCU_EXPORT.exists():
        return None, None
    try:
        with NCU_EXPORT.open(newline="") as fh:
            rows = list(csv.reader(fh))
        header = next(r for r in rows if "Kernel Name" in r)
        units = rows[rows.index(header) + 1]
        k, rd, wr = header.index("Kernel Name"), header.index("dram__bytes_read.sum"), header.index("dram__bytes_write.sum")
        scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
        totals = []
        for r in rows[rows.index(header) + 2 :]:
            if len(r) > max(k, rd, wr) and kernel_substring in r[k]:
                totals.append(float(r[rd].replace(",", "")) * scale.get(units[rd], 1.0) + float(r[wr].replace(",", "")) * scale.get(units[wr], 1.0))
        if not totals:
            return None, None
        return statistics.median(totals), str(NCU_EXPORT.relative_to(REPO))
    except Exception as e:  # a malformed export must not take the bench down
        log("ncu export unreadable:", e)
        return None, None


def build_workload():
    from anemoi_transform_b200 import synthetic as syn

    t_lat, t_lon = syn.n320_like()
    data, idx, ptr, shape = syn.bilinear_matrix(0.25, t_lat, t_lon)
    n_src_ref = int(np.unique(idx).size)
    return dict(data=data, idx=idx, ptr=ptr, shape=shape, n_src_ref=n_src_ref, t_lat=t_lat, t_lon=t_lon)


def algorithmic_bytes(w, n_fields: int) -> int:
    """SURVEY §8(d): every referenced X row read once, every Y row written once, CSR read once."""
    return 4 * n_fields * (w["n_src_ref"] + w["shape"][0]) + 8 * int(w["data"].size) + 4 * (w["shape"][0] + 1)


DUMP_FIELDS, DUMP_POINTS = 12, 2048  # 26.0 MB + 25.6 MB of the 6.77 GB output at N = 1


def dump_outputs(out_dir: str, Y) -> None:
    """A fixed, seeded sample of the resident leg's output Y [target points x fields] as .npy:
    whole fields (every target point) and every field at a set of target points."""
    import torch

    n_tgt, n_cols = Y.shape
    rng = np.random.default_rng(0)
    fields = np.sort(rng.choice(n_cols, size=min(DUMP_FIELDS, n_cols), replace=False))
    points = np.sort(rng.choice(n_tgt, size=min(DUMP_POINTS, n_tgt), replace=False))
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    np.save(out / "spmm_fields.npy", Y[:, torch.from_numpy(fields).to(Y.device)].cpu().numpy())
    np.save(out / "spmm_points.npy", Y[torch.from_numpy(points).to(Y.device)].cpu().numpy())
    log(f"outputs written to {out}: fields {fields.tolist()}, {points.size} target points")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md).

    nvidia-smi takes ~100 ms to produce its first row, longer than a 20-step timed region, so the
    sampler is started before the warm-up and `mark()` brackets the timed region: only rows that
    arrived between the two marks (plus the first one after) are reported."""

    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index: int, period_ms: int = 10):
        self.rows, self.proc, self.gpu, self.period_ms = [], None, gpu_index, period_ms
        self.marks: list[int] = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", str(self.period_ms), "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception as e:  # nvidia-smi missing: report that rather than fail the bench
            log("clock sampler unavailable:", e)
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def wait_for_first_row(self, timeout_s: float = 5.0):
        t0 = time.perf_counter()
        while self.proc is not None and not self.rows and time.perf_counter() - t0 < timeout_s:
            time.sleep(0.01)

    def mark(self):
        self.marks.append(len(self.rows))

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        time.sleep(3 * self.period_ms / 1000.0)
        self.proc.terminate()
        lo, hi = (self.marks + [0, len(self.rows)])[:2] if len(self.marks) >= 2 else (0, len(self.rows))
        rows = self.rows[max(0, lo - 1) : hi + 1] or self.rows
        sm = [float(r[1]) for r in rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in rows if len(r) >= 9 for n, v in zip(names, r[5:9]) if v.lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm), "period_ms": self.period_ms}


def bind_to_gpu_numa_node(local_rank: int):
    """Run this rank (and allocate its pinned buffers) on the NUMA node its GPU hangs off, so
    H2D / D2H DMA does not cross the inter-socket link.  Best effort: sysfs may be hidden."""
    try:
        import torch

        p = torch.cuda.get_device_properties(local_rank)
        bus = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        node = int(Path(f"/sys/bus/pci/devices/{bus}/numa_node").read_text())
        if node < 0:
            return None
        cpus = set()
        for part in Path(f"/sys/devices/system/node/node{node}/cpulist").read_text().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if allowed:
            os.sched_setaffinity(0, allowed)
            return node
    except Exception as e:
        log("NUMA binding skipped:", e)
    return None


# ------------------------------------------------------------------ reference arm -------
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from benchmarks.cpu_reference import ReferenceArm

    w = build_workload()
    arm = ReferenceArm(w, CPU_SAMPLE_FIELDS)
    for _ in range(args.warmup):
        arm.step()
    seconds = fields = 0.0
    for _ in range(args.steps):
        s, f = arm.step()
        seconds, fields = seconds + s, fields + f
    value = fields / seconds
    info = arm.describe()
    arm.close()
    cpu = {"value": value, "unit": "fields/s", **info}
    print(
        json.dumps(
            {
                "impl": "reference",
                "metric": "regrid_fields_per_s",
                "value": value,
                "unit": "fields/s",
                "n_gpus": args.gpus,
                "steps": args.steps,
                "warmup": args.warmup,
                "ms_per_step": seconds / args.steps * 1e3,
                "higher_is_better": True,
                "scaling": "strong",
                "vs_baseline": None,
                "dtype": "f32",
                "data": "synthetic",
                "config": bench_config(args.gpus),
                "cpu_baseline": cpu,
                "e2e": {"value": value, "unit": "fields/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            }
        ),
        flush=True,
    )


# ------------------------------------------------------------------ GPU arm -------------
def cpu_baseline(w) -> dict:
    from benchmarks.cpu_reference import ReferenceArm

    arm = ReferenceArm(w, CPU_SAMPLE_FIELDS)
    times = [arm.step() for _ in range(3)]
    s, f = min(times, key=lambda t: t[0] / t[1])
    info = arm.describe()
    arm.close()
    return {"value": f / s, "unit": "fields/s", **info}


def make_fieldlist(values, lat, lon, specs=None):
    from anemoi_transform_b200 import ekd

    if specs is None:
        specs = [dict(param="t", levelist=850, step=k) for k in range(len(values))]
    return ekd.from_source("list-of-dicts", [dict(values=v, latitudes=lat, longitudes=lon, **s) for v, s in zip(values, specs)])


def plugin_e2e(w, matrix_path, n_local: int, steps: int, rank: int, barrier, max_over_ranks, page_locked: bool = False) -> dict | None:
    """FieldList of ordinary (pageable) numpy fields → RegridFilter.forward → to_numpy() of
    every output.  Each field is its own numpy array, as a decoder would deliver them.
    `page_locked`: the same call on fields whose arrays a decoder allocated with
    `device.pinned_empty` (numpy arrays in page-locked memory): no staging copy, H2D in place."""
    from anemoi_transform_b200 import synthetic as syn
    from anemoi_transform_b200.device import HostIO, pinned_fields
    from anemoi_transform_b200.filters import create_filter_by_name

    n_tgt, n_src = w["shape"]
    s_lat, s_lon = syn.regular_latlon(0.25)
    rng = np.random.default_rng(99 + rank)
    base = rng.standard_normal((min(64, n_local), n_src), dtype=np.float32)
    if page_locked:
        values, _ = pinned_fields(n_local, n_src, np.float32)
        if max_over_ranks(1.0 if values is None else 0.0) > 0.0:  # every rank or none: barriers follow
            return None
        for k, v in enumerate(values):
            v[:] = base[k % base.shape[0]]
    else:
        values = [np.array(base[k % base.shape[0]]) for k in range(n_local)]
    fl = make_fieldlist(values, s_lat, s_lon)
    regrid = create_filter_by_name("regrid", matrix=matrix_path)

    def once():
        out = regrid.forward(fl)
        return [f.to_numpy() for f in out]

    arrays = once()  # warm-up: pins the staging slots and grows the page-locked pool
    del arrays
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        arrays = None  # the consumer is done with the previous step's results
        arrays = once()
    seconds = max_over_ranks(time.perf_counter() - t0) / steps
    parity = None
    if rank == 0:
        from scipy.sparse import csr_array

        m = csr_array((w["data"], w["idx"], w["ptr"]), shape=w["shape"])
        parity = all(bool(np.array_equal((m @ values[f]).view(np.uint32), arrays[f].view(np.uint32))) for f in (0, n_local // 2, n_local - 1))
    io = HostIO.get()
    return {
        "seconds": seconds,
        "parity_spot_check": parity,
        "staging_threads": io.n_threads,
        "path": "create_filter_by_name('regrid', matrix=...).forward(FieldList of numpy fields in page-locked memory (device.pinned_empty)) + to_numpy() of every output: "
        "H2D straight from the caller's arrays -> pack -> SpMM -> unpack -> D2H straight into the page-locked arrays the caller receives"
        if page_locked
        else "create_filter_by_name('regrid', matrix=...).forward(FieldList of pageable numpy fields) + to_numpy() of every output: "
        "worker threads stage the fields into pinned slots -> H2D -> pack -> SpMM -> unpack -> D2H straight into the page-locked arrays the caller receives",
    }


class BenchGribField:
    """A GRIB-backed field as earthkit-data hands it to a filter: it owns the encoded message
    (`message()`), its `to_numpy()` decodes on the host (here through the oracle, used by the
    parity check only — the B200 path never calls it)."""

    def __init__(self, message: bytes, n_points: int, md: dict, lat, lon):
        self._message, self._n, self._md, self._lat, self._lon = message, n_points, md, lat, lon

    shape = property(lambda self: (self._n,))

    def message(self) -> bytes:
        return self._message

    def to_numpy(self, flatten: bool = False, dtype=None, index=None):
        from oracle import grib as ogrib

        v = ogrib.decode(self._message, n_points=self._n)
        return v if dtype is None else v.astype(dtype)

    def metadata(self, *keys, namespace=None, default=None, **kw):
        if namespace is not None:
            return dict(self._md) if namespace in ("mars", "default") else {}
        if not keys:
            from anemoi_transform_b200 import ekd

            return ekd.Metadata(dict(self._md))
        vals = [self._md.get(k, default) for k in keys]
        return vals[0] if len(keys) == 1 else vals

    def grid_points(self):
        return self._lat, self._lon


def grib_e2e(w, matrix_path, n_local: int, steps: int, rank: int, world: int, barrier, max_over_ranks) -> dict | None:
    """config 3 as a GRIB FieldList: 16-bit simple-packed edition-2 messages in ->
    RegridFilter.forward -> to_numpy() of every output.  The packed octets cross PCIe and are
    decoded on the device; results are float64 like the reference's (float32 matrix @ float64
    values), and float32 with `set_decode_dtype(float32)`."""
    import gc

    import psutil

    from anemoi_transform_b200 import ekd, grib
    from anemoi_transform_b200 import synthetic as syn
    from anemoi_transform_b200.device import pinned_pool_trim
    from anemoi_transform_b200.filters import create_filter_by_name
    from oracle import grib as ogrib

    n_tgt, n_src = w["shape"]
    need = n_local * (2 * n_src + 8 * n_tgt) * 1.5
    if psutil.virtual_memory().available < need:
        return None
    s_lat, s_lon = syn.regular_latlon(0.25)
    rng = np.random.default_rng(17 + rank)
    distinct = [ogrib.encode_grib2(rng.normal(280.0, 15.0, n_src), 16, 0) for _ in range(min(32, n_local))]
    # every field owns its own copy of a message, as a reader would deliver them
    messages = [bytes(bytearray(distinct[k % len(distinct)])) for k in range(n_local)]
    fields = [BenchGribField(m, n_src, dict(param="t", levelist=850, step=k), s_lat, s_lon) for k, m in enumerate(messages)]
    fl = ekd.SimpleFieldList(fields)
    regrid = create_filter_by_name("regrid", matrix=matrix_path)
    out = {}
    for name, dtype in (("float64", None), ("float32", np.float32)):
        grib.set_decode_dtype(dtype)
        try:
            gc.collect()
            pinned_pool_trim()  # the previous leg's result blocks have another size

            def once():
                return [f.to_numpy() for f in regrid.forward(fl)]

            arrays = once()
            del arrays
            barrier()
            t0 = time.perf_counter()
            for _ in range(steps):
                arrays = None
                arrays = once()
            seconds = max_over_ranks(time.perf_counter() - t0) / steps
            parity = None
            if rank == 0:
                from scipy.sparse import csr_array

                m = csr_array((w["data"], w["idx"], w["ptr"]), shape=w["shape"])
                checks = []
                for f in (0, n_local // 2, n_local - 1):
                    x = ogrib.decode(messages[f], n_points=n_src)
                    want = m @ (x if dtype is None else x.astype(dtype))
                    checks.append(bool(want.dtype == arrays[f].dtype and np.array_equal(want, arrays[f])))
                parity = all(checks)
            itemsize = arrays[0].dtype.itemsize
            del arrays
            out[name] = {
                "value": N_FIELDS / seconds,
                "unit": "fields/s",
                "ms_per_step": seconds * 1e3,
                "h2d_bytes_per_step": 2 * N_FIELDS * n_src,
                "d2h_bytes_per_step": itemsize * N_FIELDS * n_tgt,
                "parity_spot_check": parity,
            }
        finally:
            grib.set_decode_dtype(None)
    gc.collect()
    pinned_pool_trim()
    result = {
        "workload": "config 3 as a GRIB FieldList: 3120 edition-2 messages, grid-point simple packing, 16 bits per value, D = 0 (2.08 MB each)",
        "path": "create_filter_by_name('regrid', matrix=...).forward(FieldList of GRIB-backed fields) + to_numpy() of every output: "
        "packed octets staged -> H2D -> grib_unpack_kernel (decode + point-major packing) -> SpMM -> unpack -> D2H into page-locked result arrays; no host decode",
        "decode_float64": out["float64"],
        "decode_float32": out["float32"],
    }
    if rank == 0 and world == 1:
        from benchmarks.cpu_reference import grib_chain_fields_per_s

        cpu = grib_chain_fields_per_s(w, messages[: 16 * max(1, min(os.cpu_count() or 1, 32))], n_src)
        result["cpu_chain"] = cpu
        result["speedup_vs_as_is"] = out["float64"]["value"] / cpu["as_is_fields_per_s"]
        result["speedup_vs_best_effort"] = out["float64"]["value"] / cpu["best_effort_fields_per_s"]
    return result


def cabi_e2e(csr, w, n_local: int, steps: int, chunk: int, rank: int, world: int, barrier, max_over_ranks) -> dict:
    """The bare C-ABI pipeline on caller-pinned buffers: what PCIe allows for these bytes."""
    import psutil
    import torch

    from anemoi_transform_b200.device import HostPipeline

    n_tgt, n_src = w["shape"]
    per_field = 4 * (n_src + n_tgt)
    budget = 0.3 * psutil.virtual_memory().available / max(world, 1)
    pool = int(max(2 * chunk, min(n_local, budget // per_field)))
    host_in = torch.empty((pool, n_src), dtype=torch.float32).pin_memory()
    host_out = torch.empty((pool, n_tgt), dtype=torch.float32).pin_memory()
    hin = host_in.numpy()
    rng = np.random.default_rng(5 + rank)
    hin[: min(64, pool)] = rng.standard_normal((min(64, pool), n_src), dtype=np.float32)
    for f0 in range(64, pool, 64):
        hin[f0 : f0 + 64] = hin[: min(64, pool - f0)]
    fields_in = [hin[f % pool] for f in range(n_local)]
    fields_out = [host_out.numpy()[f % pool] for f in range(n_local)]
    pipe = HostPipeline(csr, chunk_fields=chunk)
    pipe.regrid(fields_in[: 2 * chunk], fields_out[: 2 * chunk])
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        pipe.regrid(fields_in, fields_out)
    torch.cuda.synchronize()
    seconds = max_over_ranks(time.perf_counter() - t0) / steps
    pipe.close()
    return {"seconds": seconds, "host_pool_fields": pool}


def pipeline_e2e(steps: int = 2, n_groups: int = 48) -> dict:
    """Config 4 through the public pipeline API, next to the reference's five-pass CPU chain."""
    import torch

    from anemoi_transform_b200 import spatial
    from anemoi_transform_b200 import synthetic as syn
    from anemoi_transform_b200.device import KnnIndex
    from anemoi_transform_b200.filters import create_filter_by_name as F
    from anemoi_transform_b200.source import FieldListSource
    from benchmarks.cpu_reference import host_cores, pipeline_chain_fields_per_s

    s_lat, s_lon = syn.octahedral(1280)
    t_lat, t_lon = syn.n320_like()
    sx, tx = spatial.latlon_to_xyz(s_lat, s_lon), spatial.latlon_to_xyz(t_lat, t_lon)
    knn = KnnIndex(sx)
    idx, dist, _ = knn.query(tuple(torch.from_numpy(a).cuda() for a in tx), k=12)
    d, i, p, shape = syn.knn_matrix(idx.cpu().numpy(), dist.cpu().numpy(), sx[0].size)
    knn.close()
    del idx, dist
    tmp = tempfile.mkdtemp(prefix="at_b200_bench_")
    path = os.path.join(tmp, "c4.npz")
    syn.save_regrid_npz(path, d, i, p, shape, s_lat, s_lon, t_lat, t_lon)
    n_src = shape[1]
    levels = [50, 100, 150, 200, 250, 300, 400, 500, 600, 700, 850, 925, 1000]
    rng = np.random.default_rng(4)
    base = {k: syn.synthetic_field(k, n_src, s) for s, k in enumerate(("u", "v", "q", "t"))}
    values, specs = [rng.uniform(0.0, 1.0, n_src).astype(np.float32)], [dict(param="lsm", levelist=0, step=0)]
    for g in range(n_groups):
        for k in ("u", "v", "q", "t"):
            values.append(np.array(base[k]))
            specs.append(dict(param=k, levelist=levels[g % 13], step=g // 13))
    fl = make_fieldlist(values, s_lat, s_lon, specs)
    filters = [
        F("regrid", matrix=path),
        F("uv_to_ddff"),
        F("q_to_r"),
        F("clip", param="r", minimum=0.0, maximum=100.0),
        F("apply_mask", mask_param="lsm", threshold=0.5, threshold_operator=">", param=["ws", "r"]),
    ]
    pipe = FieldListSource(dataset=fl)
    for f in filters:
        pipe = pipe | f

    def once():
        return [f.to_numpy() for f in pipe.forward(None)]

    out = once()
    fused = bool(getattr(pipe.execution_plan()[1], "last_forward_was_fused", False))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        out = None
        out = once()
    gpu_s = (time.perf_counter() - t0) / steps
    n_in = len(values)
    # the reference's chain on the host: one thread as it runs, and one process per core
    from scipy.sparse import csr_array

    m = csr_array((d, i, p), shape=shape)
    group = dict(u=base["u"], v=base["v"], q=base["q"], t=base["t"], level=850, lsm=values[0])
    as_is = pipeline_chain_fields_per_s(m, [group, group])
    import multiprocessing as mp

    cores = host_cores()
    _CHAIN["m"], _CHAIN["group"] = m, group
    with mp.get_context("fork").Pool(cores) as pool:
        pool.map(_chain_worker, range(cores))
        t0 = time.perf_counter()
        pool.map(_chain_worker, range(cores))
        best_effort = cores * 9 / (time.perf_counter() - t0)
    return {
        "workload": f"config 4: regrid O1280 (6,599,680 pts) -> N320-shaped, 12 nnz/row | uv_to_ddff | q_to_r | clip(r) | apply_mask(lsm > 0.5 on ws, r); {n_in} float32 fields in ({n_groups} x u,v,q,t + lsm), {len(out)} out",
        "value": n_in / gpu_s,
        "unit": "input fields/s",
        "ms_per_step": gpu_s * 1e3,
        "fused_single_launch": fused,
        "h2d_bytes_per_step": 4 * n_in * n_src,
        "d2h_bytes_per_step": 4 * len(out) * shape[0],
        "path": "FieldListSource | regrid | uv_to_ddff | q_to_r | clip | apply_mask -> Pipeline.forward -> to_numpy() of every output (ordinary numpy fields in)",
        "cpu_chain": {
            "as_is_fields_per_s": as_is,
            "as_is_cores": 1,
            "best_effort_fields_per_s": best_effort,
            "best_effort_cores": cores,
            "what": "the reference's five passes (scipy csr @ x per field, numpy wind / humidity formulas per pair, np.clip, mask) — one thread as it runs, and one process per core each running whole groups",
        },
        "speedup_vs_as_is": (n_in / gpu_s) / as_is,
        "speedup_vs_best_effort": (n_in / gpu_s) / best_effort,
    }


_CHAIN: dict = {}


def _chain_worker(_):
    from benchmarks.cpu_reference import pipeline_chain_fields_per_s

    pipeline_chain_fields_per_s(_CHAIN["m"], [_CHAIN["group"], _CHAIN["group"]])
    return 0


def run_gpu(args):
    import torch
    import torch.distributed as dist

    from anemoi_transform_b200 import _cabi
    from anemoi_transform_b200 import synthetic as syn
    from anemoi_transform_b200.device import CsrMatrix, KnnIndex
    from anemoi_transform_b200.distributed import shard_range

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        log(f"warning: --gpus {args.gpus} but WORLD_SIZE={world}; using WORLD_SIZE")
    _cabi.load(check_device=True)  # fail loudly if the CUDA library or the device is missing
    torch.cuda.set_device(local_rank)
    numa_node = bind_to_gpu_numa_node(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def all_ranks(x: float) -> list[float]:
        if world == 1:
            return [x]
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        out = torch.empty((world,), device=dev, dtype=torch.float64)
        dist.all_gather_into_tensor(out, t)
        return [float(v) for v in out.cpu()]

    w = build_workload()
    n_tgt, n_src = w["shape"]
    csr = CsrMatrix(w["data"], w["idx"], w["ptr"], w["shape"])
    lo, hi = shard_range(N_FIELDS, rank, world, 4)
    n_local = hi - lo

    def resident_leg(n_cols: int, sample_clocks: bool):
        """K launches over an [n_src, n_cols] batch resident in HBM → (ms per step on this rank, clocks, X, Y)."""
        gen = torch.Generator(device=dev).manual_seed(1234 + rank)
        X = torch.empty((n_src, n_cols), device=dev, dtype=torch.float32)
        for c0 in range(0, n_cols, 260):  # fill in slabs: randn of the whole batch would need a second copy
            X[:, c0 : c0 + 260] = torch.randn((n_src, min(260, n_cols - c0)), device=dev, dtype=torch.float32, generator=gen) * 15.0 + 280.0
        Y = torch.empty((n_tgt, n_cols), device=dev, dtype=torch.float32)
        sampler = ClockSampler(local_rank) if sample_clocks else None
        if sampler:
            sampler.start()
        for _ in range(args.warmup):
            csr.apply(X, out=Y, variant=args.variant)
        if sampler:
            sampler.wait_for_first_row()
        barrier()
        if sampler:
            sampler.mark()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(args.steps):
            csr.apply(X, out=Y, variant=args.variant)
        ev1.record()
        barrier()
        if sampler:
            sampler.mark()
        clocks = sampler.stop() if sampler else None
        return ev0.elapsed_time(ev1) / args.steps, clocks, X, Y

    # ---- device-resident, strong scaling: value + roofline ---------------------------------
    my_ms, clocks, X, Y = resident_leg(n_local, sample_clocks=(rank == 0))
    per_rank_ms = all_ranks(my_ms)
    ms_per_step = max(per_rank_ms)
    value = N_FIELDS / (ms_per_step * 1e-3)
    peak, peak_src = measured_peak_gbs()
    alg_local = algorithmic_bytes(w, n_local)
    achieved = alg_local / (per_rank_ms[0] * 1e-3) / 1e9  # rank 0's kernel: its bytes over its launch time

    # parity spot check outside the timed region (rank 0): sampled columns bit-exact vs scipy
    parity = None
    if rank == 0:
        from scipy.sparse import csr_array

        m = csr_array((w["data"], w["idx"], w["ptr"]), shape=w["shape"])
        parity = True
        for col in (0, n_local // 2 + 1, n_local - 1):
            ref = m @ X[:, col].cpu().numpy()
            parity = parity and bool(np.array_equal(ref.view(np.uint32), Y[:, col].cpu().numpy().view(np.uint32)))
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, Y)
    del X, Y
    torch.cuda.empty_cache()

    if args.value_only:
        if rank == 0:
            print(json.dumps({"metric": "regrid_fields_per_s", "value": value, "unit": "fields/s", "ms_per_step": ms_per_step, "partial": "--value-only", "roofline": {"achieved": achieved, "peak": peak, "frac": achieved / peak}, "parity_spot_check": parity}), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- weak scaling (round-1 figure): 3120 fields on every GPU ---------------------------
    weak = None
    if world > 1:
        weak_ms, _, X, Y = resident_leg(N_FIELDS, sample_clocks=False)
        weak_ms = max(all_ranks(weak_ms))
        weak = {"value": N_FIELDS * world / (weak_ms * 1e-3), "unit": "fields/s", "ms_per_step": weak_ms, "fields_per_gpu": N_FIELDS, "what": "N x 3120-field job, 3120 fields on every GPU"}
        del X, Y
        torch.cuda.empty_cache()

    # ---- kNN (config 2) ---------------------------------------------------------------------
    from anemoi_transform_b200 import spatial
    from anemoi_transform_b200.distributed import ShardedKnnQuery

    s_xyz = spatial.latlon_to_xyz(*syn.regular_latlon(0.25))
    t_xyz = spatial.latlon_to_xyz(w["t_lat"], w["t_lon"])
    t_build0 = time.perf_counter()
    knn = KnnIndex(s_xyz)
    torch.cuda.synchronize()
    knn_build_ms = (time.perf_counter() - t_build0) * 1e3
    nq = t_xyz[0].shape[0]
    sharded = ShardedKnnQuery(knn, t_xyz, k=1)
    for _ in range(3):
        sharded.step()
    barrier()
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    knn_iters = 50
    k0.record()
    for _ in range(knn_iters):
        sharded.step()
    k1.record()
    barrier()
    knn_ms = max_over_ranks(k0.elapsed_time(k1)) / knn_iters
    knn_parity = sharded.check_against_single_gpu() if world > 1 else None
    knn_info = {
        "workload": "N320-shaped targets (542,080) vs 0.25deg sources (1,038,240), k=1, float64, exact",
        "queries_per_s": nq / (knn_ms * 1e-3),
        "ms_per_query_batch": knn_ms,
        "build_ms": knn_build_ms,
        "sharding": sharded.describe(),
        "gathered_equals_single_gpu": knn_parity,
    }
    sharded.close()
    del knn

    # ---- end to end through the plugin call ---------------------------------------------------
    tmp = tempfile.mkdtemp(prefix="at_b200_bench_")
    matrix_path = os.path.join(tmp, f"c3_rank{rank}.npz")
    s_lat, s_lon = syn.regular_latlon(0.25)
    syn.save_regrid_npz(matrix_path, w["data"], w["idx"], w["ptr"], w["shape"], s_lat, s_lon, w["t_lat"], w["t_lon"])
    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    plug = plugin_e2e(w, matrix_path, n_local, e2e_steps, rank, barrier, max_over_ranks)
    chunks = -(-n_local // 60)
    e2e = {
        "value": N_FIELDS / plug["seconds"],
        "unit": "fields/s",
        "h2d_bytes_per_step": 4 * N_FIELDS * n_src,
        "d2h_bytes_per_step": 4 * N_FIELDS * n_tgt,
        "steps": e2e_steps,
        "ms_per_step": plug["seconds"] * 1e3,
        "path": plug["path"],
        "parity_spot_check": plug["parity_spot_check"],
        "gpu_launches_per_step": 3 * chunks * world,
        "staging_threads_per_rank": plug["staging_threads"],
        "host_gb_per_s": 4 * N_FIELDS * (n_src + n_tgt) / plug["seconds"] / 1e9,
        "numa_node": numa_node,
    }
    import gc

    from anemoi_transform_b200.device import pinned_pool_trim

    gc.collect()
    e2e_pinned = None
    try:  # an extra leg: it must not take the headline line down with it
        plug_pl = plugin_e2e(w, matrix_path, n_local, max(1, min(2, e2e_steps)), rank, barrier, max_over_ranks, page_locked=True)
        if plug_pl is not None:
            e2e_pinned = {
                "value": N_FIELDS / plug_pl["seconds"],
                "unit": "fields/s",
                "ms_per_step": plug_pl["seconds"] * 1e3,
                "h2d_bytes_per_step": 4 * N_FIELDS * n_src,
                "d2h_bytes_per_step": 4 * N_FIELDS * n_tgt,
                "path": plug_pl["path"],
                "parity_spot_check": plug_pl["parity_spot_check"],
            }
        del plug_pl
    except Exception as e:  # noqa: BLE001
        if world > 1:
            raise  # the other ranks are inside its barriers
        log("e2e_pinned_fields leg failed:", repr(e))
        e2e_pinned = {"error": repr(e)}
    gc.collect()
    pinned_pool_trim()
    cabi = cabi_e2e(csr, w, n_local, max(1, min(2, e2e_steps)), args.chunk, rank, world, barrier, max_over_ranks)
    e2e_cabi = {
        "value": N_FIELDS / cabi["seconds"],
        "unit": "fields/s",
        "ms_per_step": cabi["seconds"] * 1e3,
        "path": f"at_pipeline_regrid (C-ABI) on caller-pinned buffers, chunks of {args.chunk} fields, 3 streams: the PCIe floor of these bytes",
        "host_pool_fields": cabi["host_pool_fields"],
    }

    gc.collect()
    grib_leg = None
    if not args.skip_grib:
        try:  # an extra leg: it must not take the headline line down with it
            grib_leg = grib_e2e(w, matrix_path, n_local, max(1, min(2, e2e_steps)), rank, world, barrier, max_over_ranks)
        except Exception as e:  # noqa: BLE001
            if world > 1:
                raise  # the other ranks are inside its barriers
            log("e2e_grib leg failed:", repr(e))
            grib_leg = {"error": repr(e)}

    pipe4 = None
    if world == 1 and not args.skip_pipeline:
        gc.collect()
        torch.cuda.empty_cache()
        pipe4 = pipeline_e2e()

    if rank == 0:
        base = cpu_baseline(w) if world == 1 else None
        traffic, traffic_src = ncu_traffic_bytes()
        line = {
            "metric": "regrid_fields_per_s",
            "value": value,
            "unit": "fields/s",
            "n_gpus": world,
            "steps": args.steps,
            "warmup": args.warmup,
            "ms_per_step": ms_per_step,
            "higher_is_better": True,
            "scaling": "strong",
            "vs_baseline": None,
            "dtype": "f32",
            "data": "synthetic",
            "config": bench_config(world),
            "fields_per_gpu": [shard_range(N_FIELDS, r, world, 4)[1] - shard_range(N_FIELDS, r, world, 4)[0] for r in range(world)],
            "per_rank_ms": per_rank_ms,
            "spmm_variant": args.variant,
            "clocks": clocks,
            "e2e": e2e,
            "e2e_pinned_fields": e2e_pinned,
            "e2e_cabi": e2e_cabi,
            "pipeline_e2e": pipe4,
            "e2e_grib": grib_leg,
            "gpu_launches": args.steps * world,
            "roofline": {
                "bound": "hbm",
                "achieved": achieved,
                "peak": peak,
                "unit": "GB/s",
                "frac": achieved / peak,
                "traffic": traffic,
                "traffic_source": traffic_src,
                "traffic_note": "ncu capture of the N=1 launch (3120 fields)" if traffic else None,
                "kernel": f"spmm_f32_kernel (one launch per step per GPU, {n_local} fields on rank 0)",
                "algorithmic_bytes_per_launch": alg_local,
                "n_src_referenced": w["n_src_ref"],
                "peak_source": peak_src,
                "frac_of_8TBs_nominal": achieved / 8000.0,
            },
            "weak": weak,
            "cpu_baseline": base,
            "knn": knn_info,
            "parity_spot_check": parity,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def reserve_stdout():
    """Keep the process's real stdout for the one JSON line: everything else that writes to
    fd 1 (NCCL prints its version banner there, libraries may print warnings) goes to stderr."""
    sys.stdout.flush()
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = real


def positive_int(text: str) -> int:
    n = int(text)
    if n < 1:
        raise argparse.ArgumentTypeError(f"must be at least 1, got {n}")
    return n


def main():
    reserve_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument(
        "--steps",
        type=positive_int,
        default=20,
        help="timed steps of the device-resident leg (the headline value); the end-to-end legs time min(--steps, --e2e-steps) steps, the pinned, C-ABI and GRIB legs at most 2",
    )
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--variant", type=int, default=0, help="at_spmm kernel shape (0 = default)")
    ap.add_argument("--chunk", type=int, default=64, help="fields per chunk of the C-ABI host pipeline")
    ap.add_argument("--e2e-steps", type=positive_int, default=3, help="upper bound on the timed steps of the plugin-call leg")
    ap.add_argument("--skip-pipeline", action="store_true", help="skip the config-4 pipeline leg")
    ap.add_argument("--skip-grib", action="store_true", help="skip the GRIB-input leg")
    ap.add_argument("--value-only", action="store_true", help="device-resident leg only (for ncu captures); prints a partial line")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a fixed sample of the last timed step's output as DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else max(args.warmup, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
