"""The missing-aware SpMM (`at_spmm_missing`) against the plain one (`at_spmm`) on the same inputs.

Two O1280 (6 599 680 points) -> N320-like (542 080) matrices built on the device:
`structured-bilinear` (4 entries per row, the uniform-row kernels) and
`structured-conservative` (rows of varying length, the general staging path).  Three batches:
1024 and 3120 float32 fields and 1024 float64 fields (float32 weights: float64 results),
point-major in HBM, uniform in [250, 300) with a seeded land mask: about 30 % of the source
points NaN in every field but the first.  The inputs (27–82 GB) are larger than L2.

For each (matrix, batch) the plain launch and the two policies are timed alternately, three
rounds of [plain, all, heaviest], each round CUDA events over 5 launches after 2 warm-up
launches; the median round is reported.  Algorithmic bytes are those of DESIGN §3.8:
sx·F·n_src_ref + sy·F·n_tgt + (4 + sw)·nnz + 4·(n_tgt + 1) (every referenced source row read
once, every target row written once, the CSR read once), the same for every policy.  After
timing, four fields of each policy's output are checked bit for bit against
oracle/spmm_missing.py.

The card's name, power limit and max SM clock are read in the same run.  Prints one JSON
document and writes it to --out.

    python benchmarks/spmm_missing.py [--out profiles/spmm_missing_b200.json]
"""

from __future__ import annotations

import argparse
import json
import statistics
import subprocess
import sys
from pathlib import Path

import numpy as np

REPO = Path(__file__).resolve().parent.parent
sys.path[:0] = [str(REPO), str(REPO / "anemoi-transform_b200")]

HBM_PEAK_GBS = 6537.6  # measured, DESIGN §3
POLICIES = {"plain": 0, "missing-if-all-missing": 1, "missing-if-heaviest-missing": 2}


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


def land_mask(lat, lon, seed=5, fraction=0.3):
    rng = np.random.default_rng(seed)
    la, lo = np.radians(lat), np.radians(lon)
    v = np.zeros(lat.size)
    for _ in range(12):
        c_la, c_lo = np.arcsin(rng.uniform(-1, 1)), rng.uniform(0, 2 * np.pi)
        v += np.exp(-((np.cos(la) * np.cos(c_la) * np.cos(lo - c_lo) + np.sin(la) * np.sin(c_la)) - 1) ** 2 * 8)
    return v > np.quantile(v, 1 - fraction)


def bitwise_equal(a: np.ndarray, b: np.ndarray) -> bool:
    na, nb = np.isnan(a), np.isnan(b)
    if a.dtype != b.dtype or not np.array_equal(na, nb):
        return False
    view = {4: np.uint32, 8: np.uint64}[a.dtype.itemsize]
    return bool(np.array_equal(a[~na].view(view), b[~nb].view(view)))


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="1024:float32,3120:float32,1024:float64")
    ap.add_argument("--out", default=str(REPO / "profiles" / "spmm_missing_b200.json"))
    args = ap.parse_args()

    import torch

    from anemoi_transform_b200 import synthetic as syn
    from anemoi_transform_b200.device import CsrMatrix, require_cuda
    from anemoi_transform_b200.regrid_files import make_conservative_matrix, make_structured_matrix
    from oracle.spmm_missing import csr_matvec_missing

    require_cuda()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU path")
    info = card()
    s_lat, s_lon = syn.octahedral(1280)
    t_lat, t_lon = syn.n320_like()
    land = torch.from_numpy(land_mask(s_lat, s_lon)).cuda()
    matrices = {
        "structured-bilinear": make_structured_matrix(s_lat, s_lon, t_lat, t_lon, "structured-bilinear"),
        "structured-conservative": make_conservative_matrix(s_lat, s_lon, t_lat, t_lon),
    }
    legs = []
    for method, (d, i, p, shape) in matrices.items():
        csr = CsrMatrix(d, i, p, shape)
        n_tgt, n_src = shape
        n_src_ref, nnz = int(np.unique(i).size), int(d.size)
        for batch in args.batches.split(","):
            n_fields, dt = int(batch.split(":")[0]), getattr(torch, batch.split(":")[1])
            leg = {"method": method, "pair": "o1280_to_n320_like", "fields": n_fields, "field_dtype": str(dt).split(".")[-1], "n_src_ref": n_src_ref, "nnz": nnz}
            try:
                X = torch.empty((n_src, n_fields), dtype=dt, device="cuda")
                Ys = {name: torch.empty((n_tgt, n_fields), dtype=csr.result_dtype(dt), device="cuda") for name in POLICIES}
            except torch.cuda.OutOfMemoryError as e:  # the device is shared: say so rather than fail the run
                legs.append({**leg, "not_measured": f"out of device memory: {e}"})
                continue
            X.uniform_(250.0, 300.0, generator=torch.Generator(device="cuda").manual_seed(7))
            X[:, 1:][land] = float("nan")
            rounds = {name: [] for name in POLICIES}
            for _ in range(3):
                for name, code in POLICIES.items():
                    rounds[name].append(events_ms(torch, lambda: csr.apply(X, out=Ys[name], missing=code), 2, 5))
            sx, sy = X.element_size(), Ys["plain"].element_size()
            alg = sx * n_fields * n_src_ref + sy * n_fields * n_tgt + (4 + d.itemsize) * nnz + 4 * (n_tgt + 1)
            sample = [0, 1, n_fields // 2, n_fields - 1]
            xs = X[:, sample].cpu().numpy()
            ms = {name: statistics.median(r) for name, r in rounds.items()}
            for name, code in POLICIES.items():
                gbs = alg / (ms[name] * 1e-3) / 1e9
                want = csr_matvec_missing(p, i, d, xs, code)
                leg[name] = {"ms_per_launch": ms[name], "ms_rounds": rounds[name], "algorithmic_gb_per_s": gbs, "fraction_of_measured_hbm_peak": gbs / HBM_PEAK_GBS,
                             "ratio_to_plain": ms[name] / ms["plain"], "sample_matches_oracle": bitwise_equal(Ys[name][:, sample].cpu().numpy(), want)}  # fmt: skip
            leg["algorithmic_bytes"] = alg
            legs.append(leg)
            print(json.dumps(leg), file=sys.stderr, flush=True)
            del X, Ys
            torch.cuda.empty_cache()

    result = {"benchmark": "spmm_missing", "card": info, "hbm_peak_gbs_measured": HBM_PEAK_GBS, "legs": legs}
    text = json.dumps(result)
    print(text, flush=True)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(text + "\n")


if __name__ == "__main__":
    main()
