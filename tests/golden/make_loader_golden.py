"""Mint tests/golden/reference_loader.pt: a small index directory written by this package's builder, and what the
reference's own Python loader (python/fast_plaid/search/load.py:220-322) reads from it.

    python tests/golden/make_loader_golden.py <checkout of the reference fast-plaid sources>

The loader's module imports the Rust extension and the third-party fastkmeans at import time; both are stubbed, the
loader code that runs is the reference's, unmodified.  The file holds the directory's files as the builder wrote
them (without embeddings.npy, the raw documents kept for updates, which neither loader reads), the files the loader
added (its merged mmap cache) and the tensors the loader returned; tests/test_index_io.py reads the directory back
with fast_plaid_b200.index.store and compares.
"""

import importlib.util
import os
import sys
import tempfile
import types

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from util import make_docs  # noqa: E402

from fast_plaid_b200 import search  # noqa: E402

OUT = os.path.join(HERE, "reference_loader.pt")


def load_reference_loader(ref_root: str):
    py = os.path.join(ref_root, "python")
    stub = types.ModuleType("fast_plaid.fast_plaid_rust")
    pkg = types.ModuleType("fast_plaid")
    pkg.__path__ = [os.path.join(py, "fast_plaid")]
    pkg.fast_plaid_rust = stub
    srch = types.ModuleType("fast_plaid.search")
    srch.__path__ = [os.path.join(py, "fast_plaid", "search")]
    sys.modules.update({"fast_plaid": pkg, "fast_plaid.fast_plaid_rust": stub, "fast_plaid.search": srch})
    spec = importlib.util.spec_from_file_location("fast_plaid.search.load",
                                                  os.path.join(py, "fast_plaid", "search", "load.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def read_files(path: str) -> dict[str, bytes]:
    out = {}
    for name in sorted(os.listdir(path)):
        with open(os.path.join(path, name), "rb") as f:
            out[name] = f.read()
    return out


def main(ref_root: str) -> None:
    ref_load = load_reference_loader(ref_root)
    with tempfile.TemporaryDirectory() as path:
        docs = make_docs(24, 4, 16, seed=321)
        # batch_size=10: three chunks, so the loader merges chunk files
        search.FastPlaid(path, device="cpu").create(docs, kmeans_niters=2, batch_size=10, seed=7)
        files = read_files(path)
        del files["embeddings.npy"]
        ref = ref_load._load_index_tensors_cpu(index_path=path)
        added = {k: v for k, v in read_files(path).items() if k not in files and k != "embeddings.npy"}
    keep = ("nbits", "centroids", "bucket_weights", "bucket_cutoffs", "ivf", "ivf_lengths", "doc_lengths",
            "doc_codes", "doc_residuals")
    reference = {k: (ref[k].clone() if torch.is_tensor(ref[k]) else ref[k]) for k in keep}
    torch.save({"source": "reference python/fast_plaid/search/load.py::_load_index_tensors_cpu, torch "
                          + torch.__version__,
                "files": files, "loader_files": added, "reference": reference}, OUT)
    print("wrote", OUT, os.path.getsize(OUT), "bytes;", len(files), "index files,", sorted(added), "added by the loader")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(sys.argv[1])
