"""Mint tests/golden/update_centroids_ref.pt by running the reference's own ``update_centroids``
(python/fast_plaid/search/update.py:65-203), unmodified.

    python tests/golden/make_update_golden.py <checkout of the reference fast-plaid sources>

The module imports the Rust extension, ``usearch`` and the metadata filter at import time; those are stubbed, the
code that runs is the reference's.  ``device="cpu:0"`` takes its torch distance branch (:143-150): the branch test is
a string compare with "cpu", and "cpu:0" is the same device to torch.  The k-means it calls is injected: the
oracle's Lloyd loop (oracle/index_oracle.py::kmeans), recorded with the arguments it is called with.

The index directory is written by this package's builder (without embeddings.npy, so that an update of it takes
the buffer branch).  Three cases: documents near the existing centroids (no outliers), a few shifted tokens among
them, and enough shifted tokens to span several `max_points_per_centroid` groups.  Every token's squared distance
is checked to sit clear of the squared threshold, so that the outlier set does not depend on summation order.
"""

import importlib.util
import json
import os
import shutil
import sys
import tempfile
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from util import make_docs  # noqa: E402

from fast_plaid_b200 import search  # noqa: E402
from oracle import index_oracle as io  # noqa: E402

OUT = os.path.join(HERE, "update_centroids_ref.pt")
MARGIN = 1e-3  # min | min_k |x - c_k|^2 - threshold^2 | over every token of every case


def load_reference_update(ref_root: str):
    py = os.path.join(ref_root, "python")
    rust = types.ModuleType("fast_plaid.fast_plaid_rust")
    pkg = types.ModuleType("fast_plaid")
    pkg.__path__ = [os.path.join(py, "fast_plaid")]
    pkg.fast_plaid_rust = rust
    srch = types.ModuleType("fast_plaid.search")
    srch.__path__ = [os.path.join(py, "fast_plaid", "search")]
    filt = types.ModuleType("fast_plaid.filtering")
    filt.update = lambda **kw: None
    us = types.ModuleType("usearch")
    us_index = types.ModuleType("usearch.index")
    us_index.Index = None  # only the device == "cpu" branch uses it
    sys.modules.update({"fast_plaid": pkg, "fast_plaid.fast_plaid_rust": rust, "fast_plaid.search": srch,
                        "fast_plaid.filtering": filt, "usearch": us, "usearch.index": us_index})
    mods = {}
    for name in ("load", "update"):
        spec = importlib.util.spec_from_file_location(f"fast_plaid.search.{name}",
                                                      os.path.join(py, "fast_plaid", "search", f"{name}.py"))
        mod = importlib.util.module_from_spec(spec)
        sys.modules[spec.name] = mod
        spec.loader.exec_module(mod)
        mods[name] = mod
    return mods["update"]


def oracle_kmeans(outliers: torch.Tensor, k: int, niters: int, seed: int, mppc: int) -> torch.Tensor:
    """compute_kmeans (fast_plaid.py:107-185) for a tensor of outlier rows, with the oracle's Lloyd loop: every row
    is a sample (fewer than 1 + 16 sqrt(120 n) rows), K = min(k, rows), L2-normalised fp16 centroids."""
    data = outliers.to(torch.float16)
    c = io.kmeans(data, min(k, data.shape[0]), niters, seed, mppc)
    return torch.nn.functional.normalize(c.float(), dim=-1).half()


def near_centroid_docs(centroids: torch.Tensor, n_docs: int, lo: int, hi: int, g: torch.Generator):
    docs = []
    for _ in range(n_docs):
        n = int(torch.randint(lo, hi + 1, (1,), generator=g))
        c = centroids[torch.randint(0, centroids.shape[0], (n,), generator=g)].float()
        docs.append(torch.nn.functional.normalize(c + 0.01 * torch.randn(n, c.shape[1], generator=g), dim=-1))
    return docs


def shifted_tokens(n: int, dim: int, g: torch.Generator) -> torch.Tensor:
    """Tokens from a region the codebook never saw: a handful of new directions, the first dimension pushed up."""
    centers = torch.randn(4, dim, generator=g)
    centers[:, 0] += 6.0
    x = centers[torch.randint(0, 4, (n,), generator=g)] + 0.3 * torch.randn(n, dim, generator=g)
    return torch.nn.functional.normalize(x, dim=-1)


def read_files(path: str) -> dict[str, bytes]:
    out = {}
    for name in sorted(os.listdir(path)):
        with open(os.path.join(path, name), "rb") as f:
            out[name] = f.read()
    return out


def main(ref_root: str) -> None:
    torch.set_num_threads(1)  # the fixture must not depend on the blocking of a threaded GEMM
    ref_update = load_reference_update(ref_root)
    base_docs = make_docs(40, 10, 20, seed=515)
    with tempfile.TemporaryDirectory() as tmp:
        base = os.path.join(tmp, "base")
        search.FastPlaid(base, device="cpu").create(base_docs, kmeans_niters=2, seed=3)
        os.remove(os.path.join(base, "embeddings.npy"))
        files = read_files(base)
        centroids = torch.from_numpy(np.load(os.path.join(base, "centroids.npy")))
        threshold = float(np.load(os.path.join(base, "cluster_threshold.npy")).item())
        g = torch.Generator().manual_seed(77)
        cases = []
        for name, n_shift, mppc in (("no_outliers", 0, 256), ("few_outliers", 30, 256), ("several_groups", 150, 32)):
            docs = near_centroid_docs(centroids, 12, 8, 16, g)
            if n_shift:
                extra = shifted_tokens(n_shift, centroids.shape[1], g)
                for j, part in enumerate(torch.tensor_split(extra, 3)):
                    docs[j] = torch.cat([docs[j], part])
            flat = torch.cat(docs)
            d2 = torch.cdist(flat.double(), centroids.double()).pow(2).min(1).values
            margin = float((d2 - threshold**2).abs().min())
            assert margin > MARGIN, f"{name}: a token sits {margin:.2e} from the threshold; pick another seed"
            calls = []

            def compute_kmeans_fn(documents_embeddings, dim, device, kmeans_niters, max_points_per_centroid, seed,
                                  n_samples_kmeans=None, use_triton_kmeans=None, num_partitions=None):
                calls.append({"outliers": documents_embeddings.clone(), "num_partitions": num_partitions,
                              "kmeans_niters": kmeans_niters, "seed": seed,
                              "max_points_per_centroid": max_points_per_centroid})
                return oracle_kmeans(documents_embeddings, num_partitions, kmeans_niters, seed,
                                     max_points_per_centroid)

            work = os.path.join(tmp, name)
            shutil.copytree(base, work)
            ref_update.update_centroids(index_path=work, new_embeddings=docs, cluster_threshold=threshold,
                                        device="cpu:0", kmeans_niters=2, max_points_per_centroid=mppc, seed=11,
                                        compute_kmeans_fn=compute_kmeans_fn)
            with open(os.path.join(work, "metadata.json")) as f:
                meta = json.load(f)
            final = np.load(os.path.join(work, "centroids.npy"))  # the existing rows are kept: only new ones stored
            assert np.array_equal(final[: centroids.shape[0]].astype(np.float32), centroids.float().numpy())
            cases.append({"name": name, "docs": docs, "max_points_per_centroid": mppc, "kmeans_niters": 2, "seed": 11,
                          "calls": calls, "centroids_added": final[centroids.shape[0]:],
                          "ivf_lengths": np.load(os.path.join(work, "ivf_lengths.npy")),
                          "num_partitions": meta["num_partitions"]})
            print(f"{name}: {len(calls) and calls[0]['outliers'].shape[0]} outliers, "
                  f"k_update {calls[0]['num_partitions'] if calls else None}, K {meta['num_partitions']}, "
                  f"margin {margin:.3g}")
    torch.save({"source": "reference python/fast_plaid/search/update.py::update_centroids, device='cpu:0', torch "
                          + torch.__version__ + ", 1 thread",
                "files": files, "threshold": threshold, "cases": cases}, OUT)
    print("wrote", OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(sys.argv[1])
