"""Pixel-exact HEALPix conservative matrices (`method="healpix-conservative"`): the cost of
building them on the device and of applying them.

Four pairs: H1024 nested (12 582 912 points) -> O96 (40 320; the longest rows), O1280
(6 599 680) -> H256 (786 432), H256 -> regular 0.25° (1 038 240) and H128 -> H96 (a
non-integer nside ratio).  For each:

* device build: `healpix_count_kernel` and `healpix_fill_kernel` alone (CUDA events over 10
  launches after 2 warm-up launches), and `make_healpix_conservative_matrix` end to end (grid
  recognition of both point lists, tables, uploads, count, scan, fill, the nested column map
  and row sort, download), median of 3;
* entries per target row (min, mean, max);
* the SpMM (`at_spmm`, float32 fields point-major in HBM) at 1024 and 3120 fields: ms per launch
  from CUDA events over 10 launches after 3 warm-up launches, algorithmic bytes
  4·F·(n_src_ref + n_tgt) + 8·nnz + 4·(n_tgt + 1) and their rate as a fraction of the measured
  6 537.6 GB/s HBM copy rate (DESIGN §3).  The inputs are larger than L2.

The card's name, power limit and max SM clock are read in the same run.  Prints one JSON
document and writes it to --out.

    python benchmarks/healpix_matrix.py [--out profiles/healpix_matrix_b200.json]
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
    ap.add_argument("--out", default=str(REPO / "profiles" / "healpix_matrix_b200.json"))
    args = ap.parse_args()

    import torch

    from anemoi_transform_b200 import synthetic as syn
    from anemoi_transform_b200._cabi import call
    from anemoi_transform_b200.device import CsrMatrix, require_cuda, stream_ptr, to_device_f64
    from anemoi_transform_b200.regrid_files import _box_rows, make_healpix_conservative_matrix

    require_cuda()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU path")
    info = card()
    pairs = {
        "h1024_nested_to_o96": ((1024, 1), syn.octahedral(96)),
        "o1280_to_h256": (syn.octahedral(1280), (256, 0)),
        "h256_to_0.25deg": ((256, 0), syn.regular_latlon(0.25)),
        "h128_to_h96": ((128, 0), (96, 0)),
    }
    keep = []

    def points(g):
        return syn.healpix(g[0], "nested" if g[1] else "ring") if isinstance(g[0], int) else g

    def side(g, which):
        if isinstance(g[0], int):
            return (g[0], g[1], *[c_void_p(0)] * 5, 0, 12 * g[0] ** 2)
        t = _box_rows(*g, "healpix-conservative", which)
        if which == "target" and t[3][0] > t[3][-1]:
            t = tuple(a[::-1].copy() for a in t)
        dev = [to_device_f64(a) for a in t[:3]] + [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in t[3:]]
        keep.extend(dev)
        return (0, 0, *(c_void_p(x.data_ptr()) for x in dev), len(t[0]), int(g[0].size))

    legs, matrices = [], {}
    for name, (s, t) in pairs.items():
        (s_lat, s_lon), (t_lat, t_lon) = points(s), points(t)
        n_src, n_tgt = s_lat.size, t_lat.size
        grid = (*side(s, "source"), *side(t, "target"))
        counts = torch.empty((n_tgt,), dtype=torch.int32, device="cuda")
        count_ms = events_ms(torch, lambda: call("at_healpix_conservative_count", *grid, c_void_p(counts.data_ptr()), stream_ptr()), 2, 10)
        indptr = torch.zeros((n_tgt + 1,), dtype=torch.int32, device="cuda")
        indptr[1:] = torch.cumsum(counts, 0, dtype=torch.int32)
        nnz = int(indptr[-1])
        data = torch.empty((nnz,), dtype=torch.float32, device="cuda")
        idx = torch.empty((nnz,), dtype=torch.int32, device="cuda")
        fill_ms = events_ms(torch, lambda: call("at_healpix_conservative_fill", *grid, c_void_p(indptr.data_ptr()), nnz, c_void_p(data.data_ptr()), c_void_p(idx.data_ptr()), stream_ptr()), 2, 10)
        e2e = []
        for _ in range(3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            d, i, p, shape = make_healpix_conservative_matrix(s_lat, s_lon, t_lat, t_lon)
            e2e.append(time.perf_counter() - t0)
        same = bool(np.array_equal(np.sort(d.view(np.uint32)), np.sort(data.cpu().numpy().view(np.uint32))) and np.array_equal(p, indptr.cpu().numpy()))
        del data, idx, counts, indptr
        row_nnz = np.diff(p)
        matrices[name] = (CsrMatrix(d, i, p, shape), int(np.unique(i).size), int(d.size), n_src, n_tgt)
        legs.append({"kind": "build", "pair": name, "n_src": n_src, "n_tgt": n_tgt, "nnz": int(d.size), "count_kernel_ms": count_ms, "fill_kernel_ms": fill_ms,
                     "make_healpix_conservative_matrix_s_median": statistics.median(e2e), "make_healpix_conservative_matrix_s_all": e2e,
                     "nnz_per_row": {"min": int(row_nnz.min()), "mean": float(row_nnz.mean()), "max": int(row_nnz.max())},
                     "rows_over_1024_entries": int((row_nnz > 1024).sum()), "kernels_match_host_api": same})  # fmt: skip
        print(json.dumps(legs[-1]), file=sys.stderr, flush=True)

    for n_fields in (int(x) for x in args.fields.split(",")):
        for name, (csr, n_src_ref, nnz, n_src, n_tgt) in matrices.items():
            gen = torch.Generator(device="cuda").manual_seed(7)
            try:
                X = torch.empty((n_src, n_fields), dtype=torch.float32, device="cuda")
                Y = torch.empty((n_tgt, n_fields), dtype=torch.float32, device="cuda")
            except torch.cuda.OutOfMemoryError as e:  # the device is shared: say so rather than fail the run
                legs.append({"kind": "spmm", "pair": name, "fields": n_fields, "not_measured": f"out of device memory: {e}"})
                continue
            X.uniform_(250.0, 300.0, generator=gen)
            ms = events_ms(torch, lambda: csr.apply(X, out=Y), 3, 10)
            alg = 4 * n_fields * (n_src_ref + n_tgt) + 8 * nnz + 4 * (n_tgt + 1)
            gbs = alg / (ms * 1e-3) / 1e9
            legs.append({"kind": "spmm", "pair": name, "fields": n_fields, "n_src_ref": n_src_ref, "nnz": nnz, "ms_per_launch": ms,
                         "algorithmic_bytes": alg, "algorithmic_gb_per_s": gbs, "fraction_of_measured_hbm_peak": gbs / HBM_PEAK_GBS})  # fmt: skip
            print(json.dumps(legs[-1]), file=sys.stderr, flush=True)
            del X, Y
            torch.cuda.empty_cache()

    result = {"benchmark": "healpix_matrix", "card": info, "hbm_peak_gbs_measured": HBM_PEAK_GBS, "legs": legs}
    text = json.dumps(result)
    print(text, flush=True)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(text + "\n")


if __name__ == "__main__":
    main()
