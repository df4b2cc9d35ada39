"""Config 3 (3120 fields, 0.25° -> N320-like) through `create_filter_by_name("regrid",
matrix=...).forward(...)` plus `to_numpy()` of every output, from ONE process, with the
streamed regrid dealt to N engines (AT_B200_DEVICES = "0,1,...,N-1"; N = 1 leaves it unset,
which is the ordinary single-engine path).

Pageable numpy fields and fields in `pinned_empty` page-locked memory, N = 1, 2, 4, 8 up to the
visible GPU count; on a single GPU also two engines on it ("0,0"), which measures what the
group costs where it cannot add a PCIe link.  Each timed step ends in a synchronise of every device.  Prints one JSON
document (and writes it to --out when given).

    python benchmarks/multi_gpu_e2e.py [--steps 5] [--warmup 2] [--out results/multi_gpu_e2e.json]
"""

from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

REPO = Path(__file__).resolve().parent.parent
sys.path[:0] = [str(REPO), str(REPO / "anemoi-transform_b200")]

from bench import build_workload, make_fieldlist  # noqa: E402


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return {"nvidia_smi": [line.strip() for line in q.stdout.splitlines() if line.strip()] or q.stderr.strip()}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--fields", type=int, default=3120)
    ap.add_argument("--engines", default="1,2,4,8", help="engine counts to try (capped at the visible GPU count)")
    ap.add_argument("--out", help="also write the JSON here")
    args = ap.parse_args()
    if args.steps < 5 or args.warmup < 2:
        ap.error("at least 2 warm-up and 5 timed steps")

    import torch

    from anemoi_transform_b200 import synthetic as syn
    from anemoi_transform_b200.device import HostIO, pinned_fields
    from anemoi_transform_b200.filters import create_filter_by_name

    n_gpus = torch.cuda.device_count()
    if n_gpus < 1:
        raise SystemExit("no CUDA device: this benchmark measures the GPU path")
    settings = [",".join(str(d) for d in range(n)) for n in (int(x) for x in args.engines.split(",")) if n <= n_gpus]
    if n_gpus == 1:
        settings.append("0,0")
    w = build_workload()
    n_tgt, n_src = w["shape"]
    s_lat, s_lon = syn.regular_latlon(0.25)
    tmp = tempfile.mkdtemp(prefix="at_mgpu_")
    matrix_path = os.path.join(tmp, "c3.npz")
    syn.save_regrid_npz(matrix_path, w["data"], w["idx"], w["ptr"], w["shape"], s_lat, s_lon, w["t_lat"], w["t_lon"])
    base = np.random.default_rng(99).standard_normal((64, n_src), dtype=np.float32)
    host_bytes = args.fields * 4 * (n_src + n_tgt)

    def sync_all():
        for d in range(n_gpus):
            torch.cuda.synchronize(d)

    legs = []
    for page_locked in (False, True):
        if page_locked:
            values, _ = pinned_fields(args.fields, n_src, np.float32)
            if values is None:
                legs.append({"inputs": "pinned_empty", "skipped": "page-locked pool exhausted"})
                continue
            for k, v in enumerate(values):
                v[:] = base[k % base.shape[0]]
        else:
            values = [np.array(base[k % base.shape[0]]) for k in range(args.fields)]
        fl = make_fieldlist(values, s_lat, s_lon)
        regrid = create_filter_by_name("regrid", matrix=matrix_path)
        reference = None
        for devices in settings:
            n = devices.count(",") + 1
            if n == 1:
                os.environ.pop("AT_B200_DEVICES", None)
            else:
                os.environ["AT_B200_DEVICES"] = devices
            times, arrays = [], None
            for step in range(args.warmup + args.steps):
                arrays = None  # the consumer is done with the previous step's results
                t0 = time.perf_counter()
                arrays = [f.to_numpy() for f in regrid.forward(fl)]
                sync_all()
                if step >= args.warmup:
                    times.append(time.perf_counter() - t0)
            if reference is None:
                reference = arrays
                identical = True
            else:
                identical = all(np.array_equal(a.view(np.uint32), b.view(np.uint32)) for a, b in zip(arrays, reference))
            s = statistics.median(times)
            legs.append(
                {
                    "inputs": "pinned_empty" if page_locked else "pageable",
                    "engines": n,
                    "devices": os.environ.get("AT_B200_DEVICES", "unset"),
                    "seconds_median": s,
                    "seconds_all": times,
                    "fields_per_s": args.fields / s,
                    "host_gb_per_s": host_bytes / s / 1e9,
                    "identical_to_single_gpu": identical,
                }
            )
            print(json.dumps(legs[-1]), file=sys.stderr, flush=True)
        os.environ.pop("AT_B200_DEVICES", None)
        del fl, values, reference, arrays, regrid
    result = {
        "benchmark": "multi_gpu_e2e",
        "workload": "config 3: 3120 float32 fields 0.25° regular lat-lon -> N320-like reduced Gaussian, bilinear CSR",
        "fields": args.fields,
        "host_bytes_per_step": host_bytes,
        "visible_gpus": n_gpus,
        "card": card(),
        "host_cpus": os.cpu_count(),
        "host_cpus_usable": len(os.sched_getaffinity(0)),
        "staging_threads_single_engine": HostIO.get().n_threads,
        "legs": legs,
    }
    text = json.dumps(result)
    print(text, flush=True)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(text + "\n")


if __name__ == "__main__":
    main()
