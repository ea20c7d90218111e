"""Centroid expansion on the GPU: the nearest-centroid kernel (fpb_nearest_centroid) against fp64, FastPlaid.update on
cuda:0 against the CPU path, search on an expanded index against the oracle, and the quality the expansion buys."""

from __future__ import annotations

import math
import os
import shutil

import numpy as np
import pytest
import torch

from util import make_docs, oracle_exact_scores, ranking_consistent

from oracle import plaid_oracle as po

pytestmark = pytest.mark.gpu

# Error bound of min_dist2 = |x|^2 - 2 max_k (<x, c_k> - |c_k|^2 / 2) with fp16 inputs and fp32 arithmetic: the
# products of fp16 values are exact in fp32; a 128-term fp32 sum is within 128 u sum_i |x_i c_i| of the exact one
# (u = 2^-24), and |x|^2, |c|^2 likewise.  u is taken as 2^-22 to leave room for the tensor cores' accumulation order
# and alignment.  Per token and centroid: 128 * 2^-22 * (2 sum_i |x_i c_i| + |x|^2 + |c|^2).
U_EFF = 2.0**-22


def _bound(x: torch.Tensor, c: torch.Tensor) -> torch.Tensor:
    """Per-token bound [n] over every centroid (the largest |c| and the Cauchy-Schwarz bound of sum |x_i c_i|)."""
    xn = x.double().norm(dim=1)
    cmax = c.double().norm(dim=1).max()
    return 128 * U_EFF * (2 * xn * cmax + xn**2 + cmax**2)


def _fp64_nearest(x: torch.Tensor, c: torch.Tensor, rows: int = 1024) -> tuple[torch.Tensor, torch.Tensor]:
    """argmin / min of |x - c_k|^2 in fp64 on the fp16 values (smallest index on exact ties)."""
    xd, cd = x.double(), c.double()
    c2 = (cd**2).sum(1)
    idx, val = [], []
    for s in range(0, xd.shape[0], rows):
        b = xd[s : s + rows]
        d = (b**2).sum(1, keepdim=True) + c2[None] - 2 * b @ cd.t()
        v, i = d.min(1)
        idx.append(i)
        val.append(v)
    return torch.cat(idx), torch.cat(val)


@pytest.mark.parametrize("K", [1000, 65536 + 37])
def test_nearest_centroid_against_fp64(K, cuda_device):
    from fast_plaid_b200.engine import kmeans_assign, nearest_centroid

    g = torch.Generator().manual_seed(K)
    n = 5000 + 77  # not a multiple of 128: the last token tile is partial
    cent = (torch.randn(K, 128, generator=g) * (0.2 + torch.rand(K, 1, generator=g))).half()  # not normalised
    ties = torch.arange(0, K - 1, 97)
    cent[ties + 1] = cent[ties]  # planted ties: equal rows, the smaller id must win
    x = cent[torch.randint(0, K, (n,), generator=g)].float() + 0.3 * torch.randn(n, 128, generator=g)
    tie_ids = ties[torch.arange(200) % ties.shape[0]]
    x[:200] = cent[tie_ids].float()  # tokens sitting exactly on a tied pair
    x = x.half()
    xd, cd = x.to(cuda_device), cent.to(cuda_device)
    assign, d2 = nearest_centroid(xd, cd)
    torch.cuda.synchronize()
    ref_i, ref_d = _fp64_nearest(xd, cd)
    bound = _bound(xd, cd)
    a = assign.long()
    # min_dist2 within the fp32 accumulation bound of the fp64 minimum
    err = (d2.double() - ref_d).abs()
    assert bool((err <= bound).all()), float((err / bound).max())
    # the index equals fp64's except where another centroid is within the bound (near-ties)
    diff = (a != ref_i).nonzero().flatten()
    if diff.numel():
        xdd, cdd = xd[diff].double(), cd.double()
        got = ((xdd - cdd[a[diff]]) ** 2).sum(1)
        assert bool((got - ref_d[diff] <= 2 * bound[diff]).all())
    assert float((a == ref_i).float().mean()) > 0.99
    # exact ties go to the smaller id
    assert bool((ref_d[:200] == 0).all()) and torch.equal(a[:200], tie_ids.to(cuda_device))
    # outlier masks agree outside the band |d - threshold^2| <= bound
    thr2 = float(ref_d.median())
    outside = (ref_d - thr2).abs() > bound
    assert torch.equal((d2 > thr2)[outside], (ref_d > thr2)[outside])
    # without the distance output the kernel assigns exactly as before
    assert torch.equal(kmeans_assign(xd, cd), assign)


def test_nearest_centroid_streams_host_points(cuda_device):
    from fast_plaid_b200.engine import nearest_centroid

    g = torch.Generator().manual_seed(2)
    cent = torch.nn.functional.normalize(torch.randn(300, 128, generator=g), dim=-1).half().to(cuda_device)
    x = torch.randn(3000, 128, generator=g)
    a1, d1 = nearest_centroid(x, cent, chunk=700)
    a2, d2 = nearest_centroid(x.to(cuda_device), cent)
    torch.cuda.synchronize()
    assert torch.equal(a1, a2) and torch.equal(d1, d2)


def _shifted_docs(n: int, seed: int, n_centers: int = 40, lo: int = 20, hi: int = 40) -> list[torch.Tensor]:
    """Documents from a region the base codebook never saw: their own centres, eight dimensions pushed up."""
    g = torch.Generator().manual_seed(seed)
    centers = torch.randn(n_centers, 128, generator=g)
    centers[:, :8] += 4.0
    out = []
    for _ in range(n):
        m = int(torch.randint(lo, hi + 1, (1,), generator=g))
        x = centers[torch.randint(0, n_centers, (m,), generator=g)] + 0.5 * torch.randn(m, 128, generator=g)
        out.append(torch.nn.functional.normalize(x, dim=-1))
    return out


@pytest.fixture(scope="module")
def base_dir(tmp_path_factory, cuda_device):
    from fast_plaid_b200 import search

    path = str(tmp_path_factory.mktemp("upd") / "base")
    docs = make_docs(1500, 20, 60, seed=91)
    fp = search.FastPlaid(path, device=cuda_device)
    fp.create(docs, kmeans_niters=4, seed=5, start_from_scratch=0)
    fp.close()
    return path, docs


def _copy(base: str, dst) -> str:
    shutil.copytree(base, str(dst))
    return str(dst)


def test_gpu_update_uses_the_kernel_and_matches_the_cpu_path(base_dir, tmp_path, monkeypatch, cuda_device):
    from fast_plaid_b200 import engine, search
    from fast_plaid_b200.index import build

    base, _ = base_dir
    new = _shifted_docs(120, 3)
    seen = {"kernel": 0}
    real_nc = engine.nearest_centroid

    def spy_nc(*a, **kw):
        seen["kernel"] += 1
        return real_nc(*a, **kw)

    monkeypatch.setattr(engine, "nearest_centroid", spy_nc)
    real_km = build.compute_kmeans
    runs = {}
    for dev in (cuda_device, "cpu"):
        calls = []

        def spy_km(docs, *a, calls=calls, **kw):
            calls.append((int(docs.shape[0]), kw["num_partitions"]))
            return real_km(docs, *a, **kw)

        monkeypatch.setattr(build, "compute_kmeans", spy_km)
        path = _copy(base, tmp_path / dev.replace(":", "_"))
        fp = search.FastPlaid(path, device=dev)
        fp.update(new, buffer_size=100, max_points_per_centroid=64)
        fp.close()
        runs[dev] = calls
    assert seen["kernel"] == 1  # the CUDA run searched the outliers on fpb_nearest_centroid, the CPU run did not
    (n_gpu, k_gpu), = runs[cuda_device]
    (n_cpu, k_cpu), = runs["cpu"]
    # tokens inside the fp32 band around threshold^2 may classify differently
    cent = torch.from_numpy(np.load(os.path.join(base, "centroids.npy"))).to(cuda_device)
    thr = float(np.load(os.path.join(base, "cluster_threshold.npy")).item())
    x = torch.cat(new).half().to(cuda_device)
    _, ref_d = _fp64_nearest(x, cent)
    n_band = int(((ref_d - thr**2).abs() <= _bound(x, cent)).sum())
    assert abs(n_gpu - n_cpu) <= n_band
    assert k_gpu == max(1, 4 * math.ceil(n_gpu / 64))
    if n_band == 0:
        assert (n_gpu, k_gpu) == (n_cpu, k_cpu)


@pytest.fixture(scope="module")
def expanded(base_dir, tmp_path_factory, cuda_device):
    """The base index after 200 shifted documents with buffer_size=100, then the documents of one new centroid
    deleted so that its inverted list is empty."""
    from fast_plaid_b200 import search
    from fast_plaid_b200.index import store

    base, docs = base_dir
    path = _copy(base, tmp_path_factory.mktemp("exp") / "idx")
    new = _shifted_docs(200, 4)
    fp = search.FastPlaid(path, device=cuda_device)
    k0 = store.read_metadata(path)["num_partitions"]
    fp.update(new[:60], buffer_size=100)
    fp.update([d.to(cuda_device) for d in new[60:]], buffer_size=100)  # the buffer comes back from disk on the host
    meta = store.read_metadata(path)
    assert meta["num_partitions"] > k0 and meta["num_documents"] == len(docs) + len(new)
    data = store.read_index(path)
    lens = data.ivf_lengths.long()
    c = k0 + int(torch.argmin(torch.where(lens[k0:] > 0, lens[k0:], 10**9)))
    off = int(lens[:c].sum())
    victims = data.ivf[off : off + int(lens[c])].tolist()
    fp.delete(victims)
    fp.close()
    return path, k0, c


def test_search_on_an_expanded_index_matches_the_oracle(expanded, cuda_device):
    from fast_plaid_b200 import search
    from fast_plaid_b200.engine import FPB_FLAG_APPROX_EXACT_ALL, DeviceIndex
    from fast_plaid_b200.index import store

    path, k0, emptied = expanded
    data = store.read_index(path)
    K = int(data.centroids.shape[0])
    assert K % 128 != 0 and K > k0
    assert int(data.ivf_lengths[emptied]) == 0 and int((data.ivf_lengths == 0).sum()) >= 1
    oidx = po.OracleIndex(data.nbits, data.centroids, data.bucket_weights, data.ivf, data.ivf_lengths.long(),
                          data.doc_codes, data.doc_residuals, data.doc_lengths)
    fp = search.FastPlaid(path, device=cuda_device)
    didx = fp.indices[cuda_device]
    g = torch.Generator().manual_seed(8)
    n_docs, Q, top_k = data.num_documents, 32, 20
    src = torch.randint(0, n_docs, (8,), generator=g).tolist()
    src[:4] = [n_docs - 1 - i * 17 for i in range(4)]  # half the queries come from the appended documents
    embs = didx.reconstruct(src)
    queries = torch.stack([torch.nn.functional.normalize(
        e.float().cpu()[torch.randint(0, e.shape[0], (Q,), generator=g)] + 0.1 * torch.randn(Q, 128, generator=g),
        dim=-1) for e in embs])
    params = DeviceIndex.make_params(top_k, 256, 8)
    st = didx.run_stages(queries.half().to(cuda_device), DeviceIndex.with_flags(params, FPB_FLAG_APPROX_EXACT_ALL))
    torch.cuda.synchronize()
    for b in range(queries.shape[0]):
        S_b = st["S"][b, :, :Q].cpu().contiguous()
        ref = po.search_one(queries[b], oidx, 8, 2000, 256, top_k, ties="canonical", return_stages=True,
                            inject={"S": S_b})
        cells = torch.unique(st["cells"][b].cpu().flatten().long())
        assert torch.equal(cells[cells >= 0], ref["cells"]), f"query {b}: probed cells differ"
        n = int(st["n_cand"][b])
        assert torch.equal(st["cand"][b, :n].cpu().long(), ref["candidates"]), f"query {b}: candidates differ"
        assert torch.equal(st["approx"][b, :n].cpu(), ref["approx"]), f"query {b}: approximate scores differ"
        r = int(st["n_rerank"][b])
        assert torch.equal(st["rerank"][b, :r].cpu().long(), ref["rerank"]), f"query {b}: pruned list differs"
        cnt = int(st["counts"][b])
        ok, why = ranking_consistent(st["ids"][b, :cnt].cpu().tolist(), st["scores"][b, :cnt].cpu().tolist(),
                                     dict(zip(ref["rerank"].tolist(), ref["exact"].tolist())), 1e-3,
                                     fallback=lambda d, b=b: float(oracle_exact_scores(oidx, queries[b], [d])[0]))
        assert ok, f"query {b}: {why}"
    res = fp.search(queries, top_k=top_k)
    assert [r[0][0] for r in res[:4]] == src[:4]
    fp.close()


def test_two_shards_on_an_expanded_index_equal_the_unsharded_search(expanded, cuda_device):
    from fast_plaid_b200.engine import DeviceIndex, shard_tensors
    from fast_plaid_b200.index import store

    path, _, _ = expanded
    data = store.read_index(path)
    didx = DeviceIndex(data, cuda_device)
    g = torch.Generator().manual_seed(9)
    Q = 32
    q16 = torch.nn.functional.normalize(torch.randn(12, Q, 128, generator=g), dim=-1).half().to(cuda_device)
    params = DeviceIndex.make_params(20, 256, 8)
    ids, scores, counts = didx.search(q16, params)
    shards = []
    for r in range(2):
        sh, base = shard_tensors(data, r, 2)
        shards.append(DeviceIndex(sh, cuda_device, doc_id_base=base))
    all_keys = torch.stack([d.shard_approx_keys(q16, params) for d in shards])
    recs = torch.stack([d.shard_exact_records(all_keys, r, Q, params) for r, d in enumerate(shards)])
    i2, s2, c2 = didx.merge_records(recs, 20)
    torch.cuda.synchronize()
    assert torch.equal(i2, ids) and torch.equal(s2, scores) and torch.equal(c2, counts)


def test_expansion_improves_reconstruction_and_retrieval(base_dir, tmp_path, cuda_device):
    """200 shifted documents added with buffer_size=100 (expansion) and with buffer_size=10**9 (control, the codebook
    stays as it was): the expanded codebook reconstructs them better and finds them at least as often."""
    from fast_plaid_b200 import search

    base, docs = base_dir
    new = _shifted_docs(200, 6)
    ids = list(range(len(docs), len(docs) + len(new)))
    g = torch.Generator().manual_seed(10)
    picks = ids[::5]
    queries = torch.stack([torch.nn.functional.normalize(
        new[d - len(docs)][torch.randint(0, new[d - len(docs)].shape[0], (16,), generator=g)]
        + 0.05 * torch.randn(16, 128, generator=g), dim=-1) for d in picks])
    out = {}
    for name, bs in (("expanded", 100), ("control", 10**9)):
        fp = search.FastPlaid(_copy(base, tmp_path / name), device=cuda_device)
        fp.update(new, buffer_size=bs)
        emb = fp.get_embeddings(ids)
        cos = torch.cat([(e.float() * s).sum(1) for e, s in zip(emb, new)])
        res = fp.search(queries, top_k=5)
        out[name] = (float(cos.mean()), sum(int(r[0][0] == d) for r, d in zip(res, picks)))
        fp.close()
    print(f"[expansion] mean cosine, top-1 hits: {out}")
    assert out["expanded"][0] > out["control"][0]
    assert out["expanded"][1] >= out["control"][1]
