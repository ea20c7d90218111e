"""Mint tests/golden/kmeans_ref.pt and kmeans_ref_fresh.pt by running the REFERENCE's own k-means code.

The Lloyd loop the reference layers on the (absent) third-party `fastkmeans` package lives in
python/fast_plaid/search/kmeans.py:60-223 of the reference and is plain PyTorch.  This script
imports that file unmodified -- only `fastkmeans` itself is stubbed with an empty base class --
seeds the RNG exactly as `FastKMeans.train` does (kmeans.py:236-238) and records inputs and
outputs.  tests/test_oracle.py then requires oracle/index_oracle.py::kmeans to reproduce the
recorded centroids, which pins that part of the oracle on reference outputs.

    python tests/golden/make_kmeans_golden.py <checkout of the reference fast-plaid sources>
"""

import importlib.util
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "kmeans_ref.pt")
OUT_FRESH = os.path.join(HERE, "kmeans_ref_fresh.pt")


def load_reference_kmeans(ref_root: str):
    stub = types.ModuleType("fastkmeans")

    class FastKMeans:  # the third-party base class; never instantiated here
        pass

    stub.FastKMeans = FastKMeans
    sys.modules.setdefault("fastkmeans", stub)
    path = os.path.join(ref_root, "python", "fast_plaid", "search", "kmeans.py")
    spec = importlib.util.spec_from_file_location("ref_kmeans", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def run_case(mod, data_f16: torch.Tensor, k: int, niters: int, seed: int, mppc: int):
    # FastKMeans.train (kmeans.py:236-241): seeds, then norms in the data's own dtype
    torch.manual_seed(seed)
    np.random.seed(seed)
    norms = (data_f16**2).sum(dim=1)
    centroids, labels = mod._kmeans_torch_double_chunked(
        data_f16, norms, k=k, device=torch.device("cpu"), dtype=None, max_iters=niters, tol=1e-8,
        chunk_size_data=51_200, chunk_size_centroids=10_240, max_points_per_centroid=mppc, use_triton=False)
    return centroids, labels


def main(ref_root: str):
    torch.set_num_threads(1)  # the fixture must not depend on the blocking of a threaded GEMM
    mod = load_reference_kmeans(ref_root)
    g = torch.Generator().manual_seed(2024)
    cases = []
    # (n, dim, k, niters, seed, max_points_per_centroid)
    for n, dim, k, niters, seed, mppc in [(3000, 32, 64, 4, 42, 256),     # plain
                                          (2600, 64, 8, 4, 7, 256),       # subsampling: n > k*mppc
                                          (600, 16, 256, 3, 11, 256)]:    # many clusters -> empty-cluster reseed
        mix = torch.randn(k if k < 100 else 20, dim, generator=g)
        x = mix[torch.randint(0, mix.shape[0], (n,), generator=g)] + 0.3 * torch.randn(n, dim, generator=g)
        x = torch.nn.functional.normalize(x, dim=-1).half()
        c, labels = run_case(mod, x, k, niters, seed, mppc)
        cases.append(dict(data=x, k=k, niters=niters, seed=seed, max_points_per_centroid=mppc,
                          centroids=c, labels=labels))
        print(f"n={n} dim={dim} k={k}: centroids {tuple(c.shape)}, empty-safe, labels {tuple(labels.shape)}")
    torch.save({"source": "reference python/fast_plaid/search/kmeans.py::_kmeans_torch_double_chunked, "
                          "torch " + torch.__version__ + ", CPU, 1 thread",
                "cases": cases}, OUT)
    print("wrote", OUT, os.path.getsize(OUT), "bytes")
    # a problem drawn apart from the mixtures above: plain normalised noise
    g = torch.Generator().manual_seed(99)
    x = torch.nn.functional.normalize(torch.randn(1500, 24, generator=g), dim=-1).half()
    k, niters, seed, mppc = 32, 3, 5, 256
    c, _ = run_case(mod, x, k, niters, seed, mppc)
    torch.save({"source": "reference python/fast_plaid/search/kmeans.py::_kmeans_torch_double_chunked, "
                          "torch " + torch.__version__ + ", CPU, 1 thread",
                "case": dict(data=x, k=k, niters=niters, seed=seed, max_points_per_centroid=mppc, centroids=c)},
               OUT_FRESH)
    print("wrote", OUT_FRESH, os.path.getsize(OUT_FRESH), "bytes")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(sys.argv[1])
