#!/usr/bin/env python
"""Config 3 as complex-packed GRIB2 messages with second-order spatial differencing (template
5.3) against the simple-packed messages of the same X, through the plugin call (regrid.forward +
to_numpy), float64 and float32 decode, the two packings alternated in the same process.

Fields: N_FIELDS (default 3 120) edition-2 messages of smooth synthetic fields on the 0.25°
grid (1 038 240 points, 16 bits, seeded): 32 distinct fields, each message its own copy; the
5.3 messages use groups of 16 values.  Reports section-7 octets and bits per value, fields/s,
the octets that cross PCIe per call, and from `torch.profiler` (in a pass of its own) the
device time and launch count of the complex kernels, grib_unpack_kernel and the host-to-device
copies of one upload of all fields.  The GPU's name, power limit and clock are read in the
same run.

    python benchmarks/grib_complex_e2e.py [--out profiles/grib_complex_b200.json]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
from pathlib import Path

REPO = Path(__file__).resolve().parent.parent
for p in (str(REPO), str(REPO / "anemoi-transform_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from anemoi_transform_b200 import _cabi, ekd, grib  # noqa: E402
from anemoi_transform_b200 import synthetic as syn  # noqa: E402
from anemoi_transform_b200.device import HostIO, pinned_pool_trim  # noqa: E402
from anemoi_transform_b200.filters import create_filter_by_name  # noqa: E402
from oracle import grib as ogrib  # noqa: E402
from oracle import grib_complex as ogx  # noqa: E402

KERNELS = ("complex_groups_kernel", "complex_tile_sums_kernel", "complex_carry_kernel", "complex_values_kernel", "grib_unpack_kernel")


def gpu_description():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else f"{torch.cuda.get_device_name()} (nvidia-smi unavailable)"


def smooth_fields(lat, lon, n, seed=0):
    """Large-scale waves plus small-scale noise of a few packing units: what a smooth 16-bit
    model field looks like to the coder."""
    rng = np.random.default_rng(seed)
    phi, lam = np.deg2rad(lat), np.deg2rad(lon)
    out = []
    for k in range(n):
        a = rng.uniform(0.5, 1.5, 4)
        v = 250.0 + 40.0 * a[0] * np.cos(phi) + 8.0 * a[1] * np.sin(2 * lam + k) * np.cos(phi) ** 2 + 3.0 * a[2] * np.sin(5 * phi + a[3] * lam)
        out.append(v + rng.normal(0.0, 0.003, lat.size))
    return out


def profile_upload(packed):
    """Device time per kernel name and of the H2D copies over one upload of every field."""
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        b = grib.upload(packed)
        torch.cuda.synchronize()
    del b
    res = {k: {"ms": 0.0, "launches": 0} for k in (*KERNELS, "h2d_copies")}
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        dt = e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
        name = e.name
        key = next((k for k in KERNELS if k in name), None)
        if key is None and "memcpy" in name.lower() and ("htod" in name.lower() or "host to device" in name.lower()):
            key = "h2d_copies"
        if key is not None:
            res[key]["ms"] += dt / 1000.0
            res[key]["launches"] += 1
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(REPO / "profiles" / "grib_complex_b200.json"))
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    _cabi.load(check_device=True)
    n_fields = int(os.environ.get("N_FIELDS", 3120))
    w = bench.build_workload()
    n_tgt, n_src = w["shape"]
    s_lat, s_lon = syn.regular_latlon(0.25)
    tmp = tempfile.mkdtemp()
    path = os.path.join(tmp, "c3.npz")
    syn.save_regrid_npz(path, w["data"], w["idx"], w["ptr"], w["shape"], s_lat, s_lon, w["t_lat"], w["t_lon"])
    values = smooth_fields(s_lat, s_lon, 32)
    simple = [ogrib.encode_grib2(v, 16, 0) for v in values]
    distinct = {"simple": simple, "complex": [ogx.from_simple(m, order=2, group_size=16) for m in simple]}
    fields, packed = {}, {}
    for name, msgs in distinct.items():
        fields[name] = [bench.BenchGribField(bytes(bytearray(msgs[k % 32])), n_src, dict(param="t", levelist=850, step=k), s_lat, s_lon) for k in range(n_fields)]
        packed[name] = grib.packed_of(fields[name])
        assert packed[name] is not None
    out = {
        "gpu": gpu_description(),
        "n_fields": n_fields,
        "n_points": int(n_src),
        "n_targets": int(n_tgt),
        "threads": HostIO.get().n_threads,
        "host_cpus": os.cpu_count(),
        "fields": "32 distinct smooth synthetic fields, 16 bits; template 5.3, order 2, groups of 16",
        "section7_octets": {k: int(sum(ogx.scan(m)["data_length"] for m in v)) for k, v in distinct.items()},
    }
    out["bits_per_value"] = {k: 8.0 * o / (32 * n_src) for k, o in out["section7_octets"].items()}
    out["h2d_GB_per_call"] = {k: p.packed_bytes / 1e9 for k, p in packed.items()}
    # same results: the two packings decode to the same values
    regrid = create_filter_by_name("regrid", matrix=path)
    few = {k: [f.to_numpy() for f in regrid.forward(ekd.SimpleFieldList(v[:8]))] for k, v in fields.items()}
    out["same_results"] = all(np.array_equal(a, b) for a, b in zip(few["simple"], few["complex"]))
    del few
    runs = {f"{k}/{d}": [] for k in fields for d in ("float64", "float32")}
    for dtype_name, dtype in (("float64", None), ("float32", np.float32)):
        grib.set_decode_dtype(dtype)
        pinned_pool_trim()
        for k in fields:  # warm-up of every shape
            arrays = [f.to_numpy() for f in regrid.forward(ekd.SimpleFieldList(fields[k]))]
            del arrays
        for _ in range(args.reps):
            for k in fields:  # alternated
                fl = ekd.SimpleFieldList(fields[k])
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                res = regrid.forward(fl)
                arrays = [f.to_numpy() for f in res]
                t1 = time.perf_counter()
                runs[f"{k}/{dtype_name}"].append(t1 - t0)
                del arrays, res
    grib.set_decode_dtype(None)
    out["plugin_call"] = {
        key: {"best_s": min(v), "median_s": float(np.median(v)), "fields_per_s": n_fields / min(v), "runs_s": v} for key, v in runs.items()
    }
    # device time of the decode kernels and of the copies, one upload of every field (float64)
    for k in packed:
        profile_upload(packed[k])  # warm
        out[f"profile_upload_{k}"] = profile_upload(packed[k])
    prof = out["profile_upload_complex"]
    chunks = max(prof["complex_groups_kernel"]["launches"], 1)
    out["per_chunk_ms"] = {
        "chunks": chunks,
        "decode": sum(prof[k]["ms"] for k in KERNELS if k.startswith("complex_")) / chunks,
        "unpack": prof["grib_unpack_kernel"]["ms"] / max(prof["grib_unpack_kernel"]["launches"], 1),
        "h2d": prof["h2d_copies"]["ms"] / chunks,
    }
    out["complex_over_simple_fields_per_s"] = {
        d: out["plugin_call"][f"complex/{d}"]["fields_per_s"] / out["plugin_call"][f"simple/{d}"]["fields_per_s"] for d in ("float64", "float32")
    }
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(out, indent=1) + "\n")
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
