"""Structured bilinear / bicubic matrices from O1280 (6 599 680 points): the cost of building
them and of applying them.

For O1280 -> N320-like (542 080 points) and O1280 -> regular 0.25° (1 038 240 points), with
`structured-bilinear` (4 entries per target) and `structured-bicubic` (16):

* host row detection (`structured_grid_rows`), median of 3 runs;
* device build: `structured_matrix_kernel` alone (CUDA events over 10 launches after 2 warm-up
  launches) and `make_structured_matrix` end to end (row detection, uploads, kernel, download);
* the SpMM (`at_spmm`, float32 fields point-major in HBM) at 1024 and 3120 fields: ms per launch
  from CUDA events over 10 launches after 3 warm-up launches, algorithmic bytes
  4·F·(n_src_ref + n_tgt) + 8·nnz + 4·(n_tgt + 1) (every referenced source row read once, every
  target row written once, the CSR read once) and their rate as a fraction of the measured
  6 537.6 GB/s HBM peak (DESIGN §3).  The inputs (26–82 GB) are far larger than L2.

The card's name and power limit are read in the same run.  Prints one JSON document and writes
it to --out (default profiles/structured_matrix.json).

    python benchmarks/structured_matrix.py [--out profiles/structured_matrix.json]
"""

from __future__ import annotations

import argparse
import json
import statistics
import subprocess
import sys
import time
from ctypes import c_void_p
from pathlib import Path

import numpy as np

REPO = Path(__file__).resolve().parent.parent
sys.path[:0] = [str(REPO), str(REPO / "anemoi-transform_b200")]

HBM_PEAK_GBS = 6537.6  # measured, DESIGN §3
METHODS = {"structured-bilinear": 2, "structured-bicubic": 4}


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return {"nvidia_smi": [line.strip() for line in q.stdout.splitlines() if line.strip()] or q.stderr.strip()}


def events_ms(torch, fn, warmup: int, steps: int) -> float:
    for _ in range(warmup):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / steps


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--fields", default="1024,3120")
    ap.add_argument("--out", default=str(REPO / "profiles" / "structured_matrix.json"))
    args = ap.parse_args()

    import torch

    from anemoi_transform_b200 import synthetic as syn
    from anemoi_transform_b200._cabi import call
    from anemoi_transform_b200.device import CsrMatrix, require_cuda, stream_ptr, to_device_f64
    from anemoi_transform_b200.regrid_files import make_structured_matrix, structured_grid_rows

    require_cuda()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU path")
    info = card()
    s_lat, s_lon = syn.octahedral(1280)
    n_src = s_lat.size
    detect = []
    for _ in range(3):
        t0 = time.perf_counter()
        rows = structured_grid_rows(s_lat, s_lon)
        detect.append(time.perf_counter() - t0)
    tables = [to_device_f64(rows[0]), to_device_f64(rows[1])] + [torch.from_numpy(a).cuda() for a in rows[2:]]

    targets = {"n320_like": syn.n320_like(), "regular_0.25deg": syn.regular_latlon(0.25)}
    legs, matrices = [], {}
    for tname, (t_lat, t_lon) in targets.items():
        n_tgt = t_lat.size
        tlat, tlon = to_device_f64(t_lat), to_device_f64(t_lon)
        for method, stencil in METHODS.items():
            nnz = stencil * stencil
            data = torch.empty((nnz * n_tgt,), dtype=torch.float32, device="cuda")
            idx = torch.empty((nnz * n_tgt,), dtype=torch.int32, device="cuda")

            def launch():
                call("at_structured_matrix", *(c_void_p(t.data_ptr()) for t in tables), rows[0].size, n_src, stencil, c_void_p(tlat.data_ptr()), c_void_p(tlon.data_ptr()), n_tgt, c_void_p(data.data_ptr()), c_void_p(idx.data_ptr()), stream_ptr())

            kernel_ms = events_ms(torch, launch, 2, 10)
            e2e = []
            for _ in range(3):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                d, i, p, shape = make_structured_matrix(s_lat, s_lon, t_lat, t_lon, method)
                e2e.append(time.perf_counter() - t0)
            same = bool(np.array_equal(d.view(np.uint32), data.cpu().numpy().view(np.uint32)) and np.array_equal(i, idx.cpu().numpy()))
            del data, idx
            matrices[(tname, method)] = (CsrMatrix(d, i, p, shape), int(np.unique(i).size), int(d.size))
            legs.append({"kind": "build", "target": tname, "method": method, "n_tgt": n_tgt, "nnz": int(d.size), "kernel_ms": kernel_ms,
                         "make_structured_matrix_s_median": statistics.median(e2e), "kernel_matches_host_api": same})  # fmt: skip
            print(json.dumps(legs[-1]), file=sys.stderr, flush=True)

    for n_fields in (int(x) for x in args.fields.split(",")):
        gen = torch.Generator(device="cuda").manual_seed(7)
        X = Y = None
        try:
            X = torch.empty((n_src, n_fields), dtype=torch.float32, device="cuda")
            Y = torch.empty((max(t[0].size for t in targets.values()), n_fields), dtype=torch.float32, device="cuda")
        except torch.cuda.OutOfMemoryError as e:  # the device is shared: say so rather than fail the run
            legs.append({"kind": "spmm", "fields": n_fields, "not_measured": f"out of device memory: {e}"})
            continue
        X.uniform_(250.0, 300.0, generator=gen)
        for tname, (t_lat, _) in targets.items():
            y = Y[: t_lat.size]
            for method in METHODS:
                csr, n_src_ref, nnz = matrices[(tname, method)]
                ms = events_ms(torch, lambda: csr.apply(X, out=y), 3, 10)
                alg = 4 * n_fields * (n_src_ref + t_lat.size) + 8 * nnz + 4 * (t_lat.size + 1)
                gbs = alg / (ms * 1e-3) / 1e9
                legs.append({"kind": "spmm", "target": tname, "method": method, "fields": n_fields, "nnz_per_row": nnz // t_lat.size, "n_src_ref": n_src_ref,
                             "ms_per_launch": ms, "algorithmic_bytes": alg, "algorithmic_gb_per_s": gbs, "fraction_of_measured_hbm_peak": gbs / HBM_PEAK_GBS})  # fmt: skip
                print(json.dumps(legs[-1]), file=sys.stderr, flush=True)
        del X, Y, y
        torch.cuda.empty_cache()

    result = {
        "benchmark": "structured_matrix",
        "source": f"O1280 ({n_src} points, {rows[0].size} rows)",
        "card": info,
        "hbm_peak_gbs_measured": HBM_PEAK_GBS,
        "host_row_detection_s": {"median": statistics.median(detect), "all": detect},
        "legs": legs,
    }
    text = json.dumps(result)
    print(text, flush=True)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(text + "\n")


if __name__ == "__main__":
    main()
