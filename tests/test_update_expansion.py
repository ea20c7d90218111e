"""The outlier buffer and centroid expansion of FastPlaid.update (python/fast_plaid/search/update.py:65-203,
:365-445; rust/index/update.rs:277-297) on the CPU path, against the reference's own update_centroids
(tests/golden/update_centroids_ref.pt, minted by tests/golden/make_update_golden.py)."""

from __future__ import annotations

import json
import os
from datetime import date

import numpy as np
import pytest
import torch

from util import make_docs

from oracle import index_oracle as io
from oracle import update_oracle as uo

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "update_centroids_ref.pt")


@pytest.fixture(scope="module")
def golden():
    return torch.load(GOLDEN, weights_only=False)


def _restore(files: dict, path) -> str:
    os.makedirs(path, exist_ok=True)
    for name, data in files.items():
        with open(os.path.join(path, name), "wb") as f:
            f.write(data)
    return str(path)


def _golden_kmeans(case):
    """The k-means the golden run injected (make_update_golden.py::oracle_kmeans)."""
    def fn(outliers: torch.Tensor, k: int) -> torch.Tensor:
        data = outliers.to(torch.float16)
        c = io.kmeans(data, min(k, data.shape[0]), case["kmeans_niters"], case["seed"], case["max_points_per_centroid"])
        return torch.nn.functional.normalize(c.float(), dim=-1).half()
    return fn


def _meta(path: str) -> dict:
    with open(os.path.join(path, "metadata.json")) as f:
        return json.load(f)


def _doclens(path: str) -> list[int]:
    from fast_plaid_b200.index import store

    return store.read_doclens(path, int(_meta(path)["num_chunks"]))


@pytest.mark.parametrize("name", ["no_outliers", "few_outliers", "several_groups"])
def test_oracle_reproduces_the_reference_update_centroids(golden, name, tmp_path):
    case = next(c for c in golden["cases"] if c["name"] == name)
    base = _restore(golden["files"], tmp_path / "base")
    cent = np.load(os.path.join(base, "centroids.npy"))
    ivfl = np.load(os.path.join(base, "ivf_lengths.npy"))
    threads = torch.get_num_threads()
    torch.set_num_threads(1)  # as the golden run
    try:
        out = uo.update_centroids(cent, ivfl, _meta(base), case["docs"], golden["threshold"],
                                  case["max_points_per_centroid"], _golden_kmeans(case))
    finally:
        torch.set_num_threads(threads)
    flat = torch.cat(case["docs"])
    if not case["calls"]:
        assert int(out["mask"].sum()) == 0 and out["k_update"] is None
        assert out["num_partitions"] == case["num_partitions"] == cent.shape[0]
        return
    call = case["calls"][0]
    assert torch.equal(flat[out["mask"]], call["outliers"])
    assert out["k_update"] == call["num_partitions"]
    want = np.concatenate([cent, case["centroids_added"]], axis=0)
    assert out["centroids"].dtype == want.dtype and np.array_equal(out["centroids"], want)
    assert np.array_equal(out["ivf_lengths"], case["ivf_lengths"])
    assert out["num_partitions"] == case["num_partitions"]


@pytest.mark.parametrize("name", ["no_outliers", "few_outliers", "several_groups"])
def test_cpu_update_reproduces_the_reference_outliers_and_threshold(golden, name, tmp_path, monkeypatch):
    from fast_plaid_b200 import search
    from fast_plaid_b200.index import build

    case = next(c for c in golden["cases"] if c["name"] == name)
    path = _restore(golden["files"], tmp_path / "idx")
    before = _meta(path)
    calls = []
    real = build.compute_kmeans

    def spy(documents_embeddings, *args, **kwargs):
        calls.append((documents_embeddings.clone(), kwargs["num_partitions"]))
        return real(documents_embeddings, *args, **kwargs)

    monkeypatch.setattr(build, "compute_kmeans", spy)
    fp = search.FastPlaid(path, device="cpu")
    fp.update(case["docs"], kmeans_niters=case["kmeans_niters"], seed=case["seed"],
              max_points_per_centroid=case["max_points_per_centroid"], buffer_size=1)
    after = _meta(path)
    assert not os.path.exists(os.path.join(path, "buffer.npy"))
    assert after["num_documents"] == before["num_documents"] + len(case["docs"])
    cent = torch.from_numpy(np.load(os.path.join(path, "centroids.npy")))
    if case["calls"]:
        assert len(calls) == 1
        assert torch.equal(calls[0][0], case["calls"][0]["outliers"])
        assert calls[0][1] == case["calls"][0]["num_partitions"]
        assert after["num_partitions"] == cent.shape[0] == before["num_partitions"] + calls[0][1]
        assert np.load(os.path.join(path, "ivf_lengths.npy")).shape[0] == cent.shape[0]
    else:  # in-distribution documents: no outliers, the codebook is unchanged
        assert calls == []
        assert after["num_partitions"] == before["num_partitions"] == cent.shape[0]
    # threshold: update.rs:277-297 on the appended tokens and the codes written for them
    codes = torch.cat([torch.from_numpy(np.load(os.path.join(path, f"{i}.codes.npy")))
                       for i in range(before["num_chunks"], after["num_chunks"])])
    want = uo.updated_threshold(golden["threshold"], before["num_embeddings"], torch.cat(case["docs"]), cent, codes)
    got = float(np.load(os.path.join(path, "cluster_threshold.npy")).item())
    assert abs(got - want) <= 1e-6 * abs(want)


def _shifted_docs(n: int, seed: int, lo: int = 6, hi: int = 12) -> list[torch.Tensor]:
    """Documents from a region a codebook trained on make_docs never saw."""
    g = torch.Generator().manual_seed(seed)
    centers = torch.randn(3, 128, generator=g)
    centers[:, :8] += 4.0
    out = []
    for _ in range(n):
        m = int(torch.randint(lo, hi + 1, (1,), generator=g))
        x = centers[torch.randint(0, 3, (m,), generator=g)] + 0.2 * torch.randn(m, 128, generator=g)
        out.append(torch.nn.functional.normalize(x, dim=-1))
    return out


def _base_index(path: str, metadata: bool = False):
    from fast_plaid_b200 import search

    docs = make_docs(40, 6, 12, seed=61)
    fp = search.FastPlaid(path, device="cpu")
    md = [{"doc": i} for i in range(len(docs))] if metadata else None
    # start_from_scratch=0: no raw embeddings.npy, so updates take the buffer branch at once
    fp.create(docs, kmeans_niters=2, seed=3, metadata=md, start_from_scratch=0)
    return fp, docs


def _check_ivf_membership(path: str, first_doc: int) -> None:
    from fast_plaid_b200.index import store

    data = store.read_index(path)
    offs = torch.zeros(data.num_documents + 1, dtype=torch.int64)
    offs[1:] = data.doc_lengths.cumsum(0)
    ivf_offs = torch.zeros(data.ivf_lengths.shape[0] + 1, dtype=torch.int64)
    ivf_offs[1:] = data.ivf_lengths.to(torch.int64).cumsum(0)
    assert data.ivf_lengths.shape[0] == data.centroids.shape[0]
    for d in range(first_doc, data.num_documents):
        for c in data.doc_codes[offs[d] : offs[d + 1]].unique().tolist():
            assert d in data.ivf[ivf_offs[c] : ivf_offs[c + 1]].tolist(), (d, c)


def test_buffer_fills_then_expands(tmp_path):
    from fast_plaid_b200 import filtering

    path = str(tmp_path / "idx")
    fp, base = _base_index(path, metadata=True)
    cent0 = open(os.path.join(path, "centroids.npy"), "rb").read()
    batches = [_shifted_docs(30, 1), _shifted_docs(30, 2), _shifted_docs(30, 3)]
    n = len(base)
    for b in batches:
        fp.update(b, metadata=[{"doc": n + i} for i in range(len(b))], buffer_size=100)
        n += len(b)
        assert _meta(path)["num_documents"] == n
    buf = np.load(os.path.join(path, "buffer.npy"), allow_pickle=True)
    assert len(buf) == 90
    assert all(np.array_equal(buf[i], d.numpy()) for i, d in enumerate(batches[0] + batches[1] + batches[2]))
    assert open(os.path.join(path, "centroids.npy"), "rb").read() == cent0  # below buffer_size: codebook untouched
    k0 = _meta(path)["num_partitions"]

    last = _shifted_docs(20, 4)
    fp.update(last, metadata=[{"doc": n + i} for i in range(len(last))], buffer_size=100)
    n += len(last)
    meta = _meta(path)
    assert not os.path.exists(os.path.join(path, "buffer.npy"))
    assert meta["num_documents"] == n
    assert meta["num_partitions"] > k0
    assert np.load(os.path.join(path, "centroids.npy")).shape[0] == meta["num_partitions"]
    all_docs = base + batches[0] + batches[1] + batches[2] + last
    assert _doclens(path) == [int(d.shape[0]) for d in all_docs]
    rows = filtering.get(index=path)
    assert [r["_subset_"] for r in rows] == list(range(n))
    assert [r["doc"] for r in rows] == list(range(n))
    _check_ivf_membership(path, len(base))


def test_update_delete_update_keeps_counts_exact(tmp_path):
    """tests/test.py:270-330 of the reference on the buffer branch: the deleted buffered document must not come
    back as a phantom when the buffer is re-added."""
    from fast_plaid_b200 import filtering

    path = str(tmp_path / "idx")
    fp, base = _base_index(path, metadata=True)
    n0 = len(base)
    new = _shifted_docs(1, 5)
    md = [{"name": "Charlie", "category": "B", "join_date": date(2020, 3, 15)}]
    fp.update(new, metadata=md)
    assert _meta(path)["num_documents"] == len(filtering.get(index=path)) == n0 + 1
    assert len(np.load(os.path.join(path, "buffer.npy"), allow_pickle=True)) == 1
    fp.delete([n0])
    assert _meta(path)["num_documents"] == len(filtering.get(index=path)) == n0
    assert not os.path.exists(os.path.join(path, "buffer.npy"))
    fp.update(new, metadata=md)
    assert _meta(path)["num_documents"] == len(filtering.get(index=path)) == n0 + 1
    # an expansion now re-adds exactly the one buffered document
    more = _shifted_docs(3, 6)
    fp.update(more, metadata=md * 3, buffer_size=4)
    assert _meta(path)["num_documents"] == len(filtering.get(index=path)) == n0 + 4
    assert not os.path.exists(os.path.join(path, "buffer.npy"))
    assert _doclens(path)[n0:] == [int(d.shape[0]) for d in new + more]
    assert [r["_subset_"] for r in filtering.get(index=path)] == list(range(n0 + 4))


def test_update_of_a_directory_with_a_reference_buffer(tmp_path):
    """A buffer.npy written the way the reference writes it (a pickled object array of the last documents' raw
    embeddings, load.py:430-444) is consumed without losing any document outside it."""
    from fast_plaid_b200.index import store

    path = str(tmp_path / "idx")
    fp, base = _base_index(path)
    tail = _shifted_docs(10, 7)
    fp.update(tail, buffer_size=10**9)
    os.remove(os.path.join(path, "buffer.npy"))
    arr = np.empty(len(tail), dtype=object)
    for i, t in enumerate(tail):
        arr[i] = t.numpy()
    np.save(os.path.join(path, "buffer.npy"), arr, allow_pickle=True)
    before = store.read_index(path)
    n_base_tok = int(before.doc_lengths[: len(base)].sum())
    new = _shifted_docs(95, 8)
    fp.update(new, buffer_size=100)
    after = store.read_index(path)
    assert not os.path.exists(os.path.join(path, "buffer.npy"))
    assert after.num_documents == len(base) + len(tail) + len(new)
    assert after.doc_lengths.tolist() == [int(d.shape[0]) for d in base + tail + new]
    # the documents outside the buffer keep their bytes
    assert torch.equal(after.doc_codes[:n_base_tok], before.doc_codes[:n_base_tok])
    assert torch.equal(after.doc_residuals[:n_base_tok], before.doc_residuals[:n_base_tok])
    _check_ivf_membership(path, len(base))


def test_nearest_centroid_refuses_other_dims():
    """fpb_nearest_centroid handles dim 128 only and says so before any CUDA call."""
    from fast_plaid_b200 import engine

    lib = engine.load_library()
    rc = lib.fpb_nearest_centroid(0, 64, 16, None, None, None, 10, None, None, None)
    assert rc == engine.FPB_ERR_UNSUPPORTED and b"dim=128" in lib.fpb_last_error()
    rc = lib.fpb_nearest_centroid(0, 128, 16, None, None, None, 10, None, None, None)
    assert rc == engine.FPB_ERR_INVALID
