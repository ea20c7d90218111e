"""Index directory layout: the product's builder/reader against the oracle's builder and against what the
reference's own Python loader read from a directory our builder wrote."""

from __future__ import annotations

import json
import os
from io import BytesIO

import numpy as np
import pytest
import torch

from util import make_docs

from fast_plaid_b200 import search
from fast_plaid_b200.index import build, store
from oracle import index_oracle as io


@pytest.fixture(scope="module")
def built(tmp_path_factory):
    path = str(tmp_path_factory.mktemp("idx"))
    docs = make_docs(260, 8, 50, seed=321)
    fp = search.FastPlaid(path, device="cpu")
    fp.create(docs, kmeans_niters=2, batch_size=100, seed=7)
    return path, docs


def test_files_and_dtypes_follow_the_reference_layout(built):
    path, docs = built
    meta = json.load(open(os.path.join(path, "metadata.json")))
    assert set(meta) == {"num_chunks", "nbits", "num_partitions", "num_embeddings", "avg_doclen", "num_documents",
                         "compress_only"}  # create.rs:569-577
    assert meta["num_documents"] == len(docs) and meta["num_chunks"] == 3 and meta["nbits"] == 4
    assert meta["num_embeddings"] == sum(d.shape[0] for d in docs)
    assert np.load(os.path.join(path, "centroids.npy")).dtype == np.float16  # create.rs:380-384
    for f in ("bucket_cutoffs.npy", "bucket_weights.npy", "avg_residual.npy", "cluster_threshold.npy"):
        assert np.load(os.path.join(path, f)).dtype == np.float32
    assert np.load(os.path.join(path, "bucket_cutoffs.npy")).shape == (15,)
    assert np.load(os.path.join(path, "bucket_weights.npy")).shape == (16,)
    assert np.load(os.path.join(path, "ivf.npy")).dtype == np.int64  # create.rs:548-552
    assert np.load(os.path.join(path, "ivf_lengths.npy")).dtype == np.int32
    off = 0
    for i in range(3):
        c = np.load(os.path.join(path, f"{i}.codes.npy"))
        r = np.load(os.path.join(path, f"{i}.residuals.npy"))
        assert c.dtype == np.int64 and r.dtype == np.uint8 and r.shape == (c.shape[0], 64)
        cm = json.load(open(os.path.join(path, f"{i}.metadata.json")))
        assert cm["embedding_offset"] == off and cm["num_embeddings"] == c.shape[0]
        off += c.shape[0]
    assert json.load(open(os.path.join(path, "plan.json"))) == {"nbits": 4, "num_chunks": 3}


def test_builder_matches_oracle_builder_byte_for_byte(built):
    path, docs = built
    data = store.read_index(path)
    oidx, extra = io.build_index(docs, data.centroids, nbits=4, batch_size=100, seed=7)
    assert torch.equal(oidx.doc_codes, data.doc_codes)
    assert torch.equal(oidx.doc_residuals, data.doc_residuals)
    assert torch.equal(oidx.ivf, data.ivf) and torch.equal(oidx.ivf_lengths, data.ivf_lengths.long())
    assert torch.equal(oidx.bucket_weights, data.bucket_weights)
    assert torch.equal(extra["bucket_cutoffs"].half(), data.bucket_cutoffs)


def test_ivf_lists_are_sorted_unique_and_consistent(built):
    path, _ = built
    data = store.read_index(path)
    offs = torch.cat([torch.zeros(1, dtype=torch.int64), data.ivf_lengths.long().cumsum(0)])
    tok2doc = torch.repeat_interleave(torch.arange(data.num_documents), data.doc_lengths)
    for c in range(0, data.ivf_lengths.shape[0], 17):
        lst = data.ivf[offs[c]:offs[c + 1]]
        assert bool((lst[1:] > lst[:-1]).all())  # strictly ascending = sorted unique (create.rs:118-124)
        assert set(lst.tolist()) == set(tok2doc[data.doc_codes == c].tolist())


LOADER_GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "reference_loader.pt")


def _write_files(path: str, files: dict[str, bytes]) -> None:
    for name, data in files.items():
        with open(os.path.join(path, name), "wb") as f:
            f.write(data)


def test_reference_loader_reads_our_directory_identically(built, tmp_path):
    """Pin the on-disk format against the reference's OWN loader
    (python/fast_plaid/search/load.py:220-322).  tests/golden/reference_loader.pt holds a directory written by our
    builder, the tensors the reference's loader read from it and the merged mmap cache it wrote there
    (tests/golden/make_loader_golden.py); our reader must return the same tensors."""
    blob = torch.load(LOADER_GOLDEN, weights_only=False)
    # the builder still writes that directory: same files, same array dtypes (embeddings.npy is not stored)
    built_path, _ = built
    assert set(os.listdir(built_path)) - {"embeddings.npy"} == set(blob["files"])
    for name in blob["files"]:
        if name.endswith(".npy"):
            stored = np.load(BytesIO(blob["files"][name]))
            assert np.load(os.path.join(built_path, name)).dtype == stored.dtype, name
    path = str(tmp_path)
    _write_files(path, blob["files"])
    ref = blob["reference"]
    ours = store.read_index(path)
    n_tok = int(ours.doc_lengths.sum())
    assert ref["nbits"] == ours.nbits
    assert torch.equal(ref["centroids"], ours.centroids)
    assert torch.equal(ref["bucket_weights"], ours.bucket_weights)
    assert torch.equal(ref["bucket_cutoffs"], ours.bucket_cutoffs)
    assert torch.equal(ref["ivf"], ours.ivf) and torch.equal(ref["ivf_lengths"], ours.ivf_lengths)
    assert torch.equal(ref["doc_lengths"], ours.doc_lengths)
    # the reference pads the tail with (max_len - last_len) zero rows (load.py:298-300)
    assert torch.equal(ref["doc_codes"][:n_tok], ours.doc_codes)
    assert torch.equal(ref["doc_residuals"][:n_tok], ours.doc_residuals)
    assert ref["doc_codes"].shape[0] - n_tok == int(ours.doc_lengths.max() - ours.doc_lengths[-1])
    # the merged mmap cache the reference wrote does not confuse our reader
    assert {"merged_codes.npy", "merged_residuals.npy"} <= set(blob["loader_files"])
    _write_files(path, blob["loader_files"])
    again = store.read_index(path)
    assert torch.equal(again.doc_codes, ours.doc_codes)


def test_pack_buckets_is_the_reference_bit_order():
    b = torch.tensor([[0b0001, 0b1000, 0b1111, 0b0010]], dtype=torch.int32)
    # LSB-first bits of each index, big-endian packing: 1 -> 1000, 8 -> 0001, 15 -> 1111, 2 -> 0100
    assert build.pack_buckets(b, 4).tolist() == [[0b10000001, 0b11110100]]


def test_synthetic_generator_is_shard_consistent():
    from fast_plaid_b200.index.synthetic import synthetic_index

    full, _ = synthetic_index(3000, 20, device="cpu", seed=5, docs_per_chunk=700)
    a, base_a = synthetic_index(3000, 20, device="cpu", seed=5, docs_per_chunk=700, doc_range=(0, 1300))
    b, base_b = synthetic_index(3000, 20, device="cpu", seed=5, docs_per_chunk=700, doc_range=(1300, 3000))
    assert (base_a, base_b) == (0, 1300)
    assert torch.equal(torch.cat([a.doc_codes, b.doc_codes]), full.doc_codes)
    assert torch.equal(torch.cat([a.doc_residuals, b.doc_residuals]), full.doc_residuals)
    assert torch.equal(a.centroids, full.centroids)
    assert int(a.ivf_lengths.sum() + b.ivf_lengths.sum()) == int(full.ivf_lengths.sum())
