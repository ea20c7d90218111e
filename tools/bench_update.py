"""Centroid expansion on a BASELINE config-2-shaped index: 100k documents x 300 tokens built by FastPlaid.create()
(K = 65 536), then 1 000 documents from a shifted distribution added with update(buffer_size=100): 60 of them first
(they go to the buffer), then the other 940 (buffer reached: the 60 are deleted, the outliers of all 1 000 are
clustered into new centroids, the 1 000 re-added with the expanded codec).

Prints one JSON line (with `--out PATH` also written to that file) with the card and its power limit, the wall time
of each phase of the expanding update (device-synchronised), and the outlier search of that update timed alone with
CUDA events: fpb_nearest_centroid against the reference's formulation (x2 + y2 - 2 x.c in 4 096-row batches,
update.py:144-150) in fp32 and fp16, plus the agreement of their outlier masks outside the fp32 tolerance band.

    python tools/bench_update.py [--out PATH]
"""
import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from fast_plaid_b200 import engine, search  # noqa: E402
from fast_plaid_b200.index import build, store  # noqa: E402
from fast_plaid_b200.index import update as upd  # noqa: E402
from fast_plaid_b200.index.synthetic import SyntheticDocuments  # noqa: E402

PEAK_FP16_DENSE_TFLOPS = 2250.0  # NVIDIA HGX B200 data sheet, one GPU, dense FP16 (not a measured figure)
DEV = "cuda:0"


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def timed(phases: dict, key: str, fn):
    def wrapper(*a, **kw):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn(*a, **kw)
        torch.cuda.synchronize()
        phases[key] = phases.get(key, 0.0) + time.perf_counter() - t0
        return out
    return wrapper


def event_ms(fn, reps: int) -> float:
    fn()  # warm-up of this exact shape
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def reference_min_dist2(x: torch.Tensor, c: torch.Tensor, rows: int = 4096) -> torch.Tensor:
    """update.py:144-150 in the given dtype: x2 + y2 - 2 x.c per 4 096-row batch, min over the centroids."""
    y2 = torch.sum(c**2, dim=1)
    out = torch.empty(x.shape[0], dtype=x.dtype, device=x.device)
    for i in range(0, x.shape[0], rows):
        b = x[i : i + rows]
        d = torch.sum(b**2, dim=1, keepdim=True) + y2 - 2 * torch.matmul(b, c.T)
        out[i : i + rows] = torch.min(d, dim=1).values
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    out = {"card": card(), "config": {"n_docs": 100_000, "doc_len": 300, "new_docs": 1000, "buffer_size": 100,
                                      "first_update_docs": 60}}
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "cfg2")
        docs = SyntheticDocuments(100_000, 300, device=DEV, seed=11, clusters=8192)
        fp = search.FastPlaid(path, device=DEV)
        t0 = time.perf_counter()
        fp.create(docs, kmeans_niters=4, seed=42)
        torch.cuda.synchronize()
        out["create_s"] = round(time.perf_counter() - t0, 2)
        meta0 = store.read_metadata(path)
        cent0 = torch.from_numpy(np.load(os.path.join(path, "centroids.npy"))).to(DEV)
        thr0 = float(np.load(os.path.join(path, "cluster_threshold.npy")).item())
        # shifted distribution: other cluster directions than the indexed corpus
        new = list(SyntheticDocuments(1000, 300, device=DEV, seed=99, clusters=64))
        t0 = time.perf_counter()
        fp.update(new[:60], buffer_size=100)
        torch.cuda.synchronize()
        out["update_to_buffer_s"] = round(time.perf_counter() - t0, 3)

        phases: dict = {}
        patches = [(upd, "outlier_mask", "outlier_search"), (build, "compute_kmeans", "kmeans"),
                   (search.FastPlaid, "_delete_documents", "delete"), (build, "encode", "encode"),
                   (upd, "_rebuild_ivf", "ivf"), (upd, "updated_threshold", "threshold")]
        saved = [(m, n, getattr(m, n)) for m, n, _ in patches]
        for m, n, key in patches:
            setattr(m, n, timed(phases, key, getattr(m, n)))
        t0 = time.perf_counter()
        try:
            fp.update(new[60:], buffer_size=100)
            torch.cuda.synchronize()
        finally:
            for m, n, f in saved:
                setattr(m, n, f)
        out["update_expanding_s"] = round(time.perf_counter() - t0, 3)
        out["phases_s"] = {k: round(v, 4) for k, v in phases.items()}
        out["phases_note"] = ("encode includes the fp32 residual norms of the threshold update; the rest of "
                              "update_expanding_s is reading the buffer, chunk and metadata files and reloading the index")
        meta1 = store.read_metadata(path)
        out["num_partitions"] = [meta0["num_partitions"], meta1["num_partitions"]]
        out["num_documents"] = [meta0["num_documents"], meta1["num_documents"]]
        out["cluster_threshold"] = [thr0, float(np.load(os.path.join(path, "cluster_threshold.npy")).item())]
        fp.close()

    # the outlier search of the expanding update alone: 1 000 x 300 tokens against the 65 536 original centroids
    x = torch.cat(new).to(torch.float16)
    n, K = int(x.shape[0]), int(cent0.shape[0])
    flop = 2.0 * n * K * 128
    reps = 20
    ms_kernel = event_ms(lambda: engine.nearest_centroid(x, cent0), reps)
    x32, c32 = x.float(), cent0.float()
    ms_ref32 = event_ms(lambda: reference_min_dist2(x32, c32), 3)
    c16 = cent0.half()
    ms_ref16 = event_ms(lambda: reference_min_dist2(x, c16), reps)
    _, d_k = engine.nearest_centroid(x, cent0)
    d_32 = reference_min_dist2(x32, c32)
    thr2 = thr0**2
    xn = x.double().norm(dim=1)
    cmax = cent0.double().norm(dim=1).max()
    band = 128 * 2.0**-22 * (2 * xn * cmax + xn**2 + cmax**2)  # as tests/test_gpu_update.py
    outside = ((d_32.double() - thr2).abs() > band)
    m_k, m_32 = d_k > thr2, d_32 > thr2
    out["outlier_search"] = {
        "tokens": n, "centroids": K, "flop": flop, "reps": reps,
        "kernel_ms": round(ms_kernel, 3),
        "kernel_tokens_per_s": round(n / (ms_kernel / 1e3)),
        "kernel_tflops": round(flop / (ms_kernel / 1e3) / 1e12, 1),
        "kernel_share_of_datasheet_fp16_dense_2250_tflops": round(flop / (ms_kernel / 1e3) / 1e12 / PEAK_FP16_DENSE_TFLOPS, 3),
        "kernel_ms_note": "CUDA events around engine.nearest_centroid (bias, kernel, |x|^2 epilogue), device-resident tokens",
        "reference_fp32_ms": round(ms_ref32, 3),
        "reference_fp16_ms": round(ms_ref16, 3),
        "speedup_vs_reference_fp32": round(ms_ref32 / ms_kernel, 1),
        "speedup_vs_reference_fp16": round(ms_ref16 / ms_kernel, 1),
        "outliers_kernel": int(m_k.sum()), "outliers_reference_fp32": int(m_32.sum()),
        "tokens_in_band": int((~outside).sum()),
        "mask_disagreements_outside_band": int((m_k != m_32)[outside].sum()),
        "k_update": max(1, 4 * math.ceil(int(m_k.sum()) / 256)),
    }
    line = json.dumps(out)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
