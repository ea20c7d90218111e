"""CPU tests of the oracle itself: golden fixtures, the reference's own numeric relations,
an independent closed-form derivation of the residual decoder, tie-mode agreement, edge cases."""

from __future__ import annotations

import glob
import os

import numpy as np
import pytest
import torch

from util import build_oracle_index, make_docs, make_queries, oracle_exact_scores

from oracle import plaid_oracle as po

GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "small_*.pt")))


def _load_golden(path):
    blob = torch.load(path, weights_only=False)
    ix = blob["index"]
    oidx = po.OracleIndex(nbits=ix["nbits"], centroids=ix["centroids"], bucket_weights=ix["bucket_weights"],
                          ivf=ix["ivf"].long(), ivf_lengths=ix["ivf_lengths"].long(), doc_codes=ix["doc_codes"].long(),
                          doc_residuals=ix["doc_residuals"], doc_lengths=ix["doc_lengths"].long())
    return blob, oidx


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p) for p in GOLDEN])
def test_oracle_reproduces_golden(path):
    blob, oidx = _load_golden(path)
    m = blob["meta"]
    for b, exp in enumerate(blob["expected"]):
        st = po.search_one(blob["queries"][b], oidx, m["n_probe"], 2000, m["n_full"], m["top_k"], ties="canonical",
                           return_stages=True)
        assert torch.equal(st["cells"], exp["cells"])
        assert torch.equal(st["candidates"], exp["candidates"])
        assert torch.equal(st["approx"], exp["approx"])
        assert torch.equal(st["rerank"], exp["rerank"])
        assert torch.equal(st["exact"], exp["exact"])
        assert st["ids"] == exp["ids"] and st["scores"] == exp["scores"]


def _decode_closed_form(res: np.ndarray, codes: np.ndarray, centroids: torch.Tensor, weights: torch.Tensor, nbits: int):
    """Independent derivation of decompress_residuals with bit operations instead of the two
    256-entry LUTs: element j of byte b is weights[bitrev_nbits((b >> (8 - nbits*(j+1))) & mask)]
    (SURVEY.md 8(a10), Appendix B)."""
    n, pd = res.shape
    per = 8 // nbits
    mask = (1 << nbits) - 1
    idx = np.zeros((n, pd, per), dtype=np.int64)
    for j in range(per):
        v = (res.astype(np.int64) >> (8 - nbits * (j + 1))) & mask
        r = np.zeros_like(v)
        for k in range(nbits):
            r |= ((v >> k) & 1) << (nbits - 1 - k)
        idx[:, :, j] = r
    w = weights.half()[torch.from_numpy(idx.reshape(n, pd * per))]
    e = w + centroids.half()[torch.from_numpy(codes)]  # one fp16 add
    nrm = torch.sqrt((e.float() ** 2).sum(-1, keepdim=True)).half()
    return (e.float() / nrm.float()).half()


@pytest.mark.parametrize("nbits,dim", [(4, 128), (2, 128), (4, 64), (2, 64)])
def test_decompress_matches_closed_form(nbits, dim):
    g = torch.Generator().manual_seed(5)
    n, K = 400, 64
    cent = torch.nn.functional.normalize(torch.randn(K, dim, generator=g), dim=-1).half()
    w = (torch.randn(2**nbits, generator=g) * 0.05).sort().values.half()
    codes = torch.randint(0, K, (n,), generator=g)
    res = torch.randint(0, 256, (n, dim * nbits // 8), generator=g, dtype=torch.uint8)
    rev, lut = po.codec_luts(nbits)
    got = po.decompress_residuals(res, w, rev, lut, codes, cent, dim, nbits)
    ref = _decode_closed_form(res.numpy(), codes.numpy(), cent, w, nbits)
    # identical up to the fp32 accumulation order inside ATen's norm (<= 1 fp16 ulp, rare)
    diff = (got.float() - ref.float()).abs()
    assert float(diff.max()) <= 2.0 ** -10
    assert float((diff > 0).float().mean()) < 5e-3


def test_pack_unpack_roundtrip():
    """Bucket indices -> create.rs packing -> the decoder's index recovery."""
    from oracle import index_oracle as io

    g = torch.Generator().manual_seed(3)
    for nbits in (2, 4):
        buckets = torch.randint(0, 2**nbits, (50, 128), generator=g, dtype=torch.int32)
        b = buckets.unsqueeze(-1).expand(50, 128, nbits).bitwise_right_shift(torch.arange(nbits, dtype=torch.int8)) & 1
        packed = io.packbits(b.flatten()).reshape(50, 128 * nbits // 8)
        rev, lut = po.codec_luts(nbits)
        idx = lut[rev[packed.flatten().long()].long()].reshape(50, 128)
        assert torch.equal(idx.to(torch.int32), buckets)


@pytest.fixture(scope="module")
def small():
    docs = make_docs(200, 10, 60, seed=77)
    oidx, _ = build_oracle_index(docs)
    queries = make_queries(5, 24, seed=78, docs=docs)
    return docs, oidx, queries


def test_reference_relations_token_scores(small):
    """tests/test.py:143-197 of the reference: search == search_token_scores rankings, and
    manual max(dim=1).sum() of the token matrix reproduces the score."""
    docs, oidx, queries = small
    for b in range(queries.shape[0]):
        a_ids, a_sc = po.search_one(queries[b], oidx, top_k=10, n_full_scores=128)
        st = po.search_one(queries[b], oidx, top_k=10, n_full_scores=128, return_stages=True)
        assert a_ids == st["ids"]
        assert all(abs(x - y) < 1e-3 for x, y in zip(a_sc, st["scores"]))
        for d, s, m in zip(st["ids"], st["scores"], st["token_matrices"]):
            assert m.shape == (queries.shape[1], int(oidx.doc_lengths[d]))  # tests/test.py:109-141
            assert abs(float(m.max(dim=1).values.float().sum()) - s) < 0.1


def test_canonical_and_torch_tie_modes_agree_up_to_ties(small):
    docs, oidx, queries = small
    for b in range(queries.shape[0]):
        t = po.search_one(queries[b], oidx, top_k=20, n_full_scores=64, ties="torch", return_stages=True)
        c = po.search_one(queries[b], oidx, top_k=20, n_full_scores=64, ties="canonical", return_stages=True)
        assert torch.equal(t["S"], c["S"])
        # same score multiset; ids may differ only inside groups of equal score
        assert sorted(t["scores"], reverse=True) == t["scores"]
        if t["ids"] != c["ids"]:
            # any doc present in one list only must be explained by an approx-score tie at the
            # pruning boundary or an exact-score tie at the top_k boundary
            only = set(t["ids"]) ^ set(c["ids"])
            sc = {d: float(oracle_exact_scores(oidx, queries[b], [d])[0]) for d in only}
            kth = min(t["scores"][-1], c["scores"][-1])
            approx_of = dict(zip(c["candidates"].tolist(), c["approx"].tolist()))
            thr = sorted(approx_of.values(), reverse=True)[min(len(approx_of), 16) - 1]
            for d in only:
                assert abs(sc[d] - kth) < 1e-6 or abs(approx_of.get(d, thr) - thr) < 1e-6


def test_scores_sorted_and_repeatable(small):
    docs, oidx, queries = small
    r1 = po.search_many(queries, oidx, top_k=15)
    r2 = po.search_many(queries, oidx, top_k=15)
    assert r1 == r2  # tests/test.py:956-974
    for res in r1:
        sc = [s for _, s in res]
        assert sc == sorted(sc, reverse=True)  # tests/test.py:939-954


def test_edge_cases(small):
    docs, oidx, queries = small
    n = len(docs)
    # top_k larger than the index: at most N results (tests/test.py:880-886)
    res = po.search_many(queries[:1], oidx, top_k=10 * n)
    assert 0 < len(res[0]) <= n
    # n_ivf_probe = 1 uses argmax (search.rs:520-521)
    assert len(po.search_many(queries[:1], oidx, top_k=5, n_ivf_probe=1)[0]) == 5
    # subset containment (tests/test.py:409-411)
    sub = list(range(0, n, 3))
    res = po.search_many(queries[:2], oidx, top_k=10, subset=[sub, sub])
    assert all(d in set(sub) for r in res for d, _ in r)
    # empty subset -> empty result (search.rs:549-551)
    assert po.search_many(queries[:1], oidx, top_k=10, subset=[[]]) == [[]]
    # non-3D queries are rejected (search.rs:234-239)
    with pytest.raises(ValueError):
        po.search_many(queries[0], oidx)
    # compress-only index (search.rs:227-232)
    bare = po.OracleIndex(oidx.nbits, oidx.centroids, oidx.bucket_weights, None, None, oidx.doc_codes,
                          oidx.doc_residuals, oidx.doc_lengths)
    with pytest.raises(ValueError, match="compress_only"):
        po.search_many(queries[:1], bare)


def test_zero_length_document_scores_like_the_reference():
    """A document with no tokens gets Q * (-10000): the fp16 value of masked_fill(-9999)."""
    docs = make_docs(40, 5, 20, seed=9)
    oidx, _ = build_oracle_index(docs)
    lens = oidx.doc_lengths.clone()
    # make document 3 empty by moving its tokens to document 4 (codes/residual rows untouched)
    lens[4] += lens[3]
    lens[3] = 0
    o2 = po.OracleIndex(oidx.nbits, oidx.centroids, oidx.bucket_weights, oidx.ivf, oidx.ivf_lengths, oidx.doc_codes,
                        oidx.doc_residuals, lens)
    q = make_queries(1, 8, seed=1)[0]
    s = oracle_exact_scores(o2, q, [3, 4])
    assert float(s[0]) == 8 * -10000.0


def test_kmeans_restatement_reproduces_reference_outputs():
    """tests/golden/kmeans_ref.pt holds inputs and OUTPUTS of the reference's own Lloyd loop
    (python/fast_plaid/search/kmeans.py:60-223, imported unmodified by
    tests/golden/make_kmeans_golden.py).  The oracle's restatement must reproduce the centroids
    bit for bit: plain run, the n > k*max_points_per_centroid subsampling path and the
    empty-cluster reseed path."""
    from oracle import index_oracle as io

    blob = torch.load(os.path.join(os.path.dirname(__file__), "golden", "kmeans_ref.pt"), weights_only=False)
    assert "reference" in blob["source"]
    assert len(blob["cases"]) == 3
    for c in blob["cases"]:
        got = io.kmeans(c["data"], c["k"], c["niters"], c["seed"], c["max_points_per_centroid"])
        assert got.shape == c["centroids"].shape
        assert torch.equal(got, c["centroids"]), float((got - c["centroids"]).abs().max())


def test_kmeans_restatement_reproduces_reference_outputs_on_fresh_data():
    """Same check on a problem drawn apart from the fixture above (plain normalised noise, k=32), recorded in
    tests/golden/kmeans_ref_fresh.pt by tests/golden/make_kmeans_golden.py."""
    from oracle import index_oracle as io

    blob = torch.load(os.path.join(os.path.dirname(__file__), "golden", "kmeans_ref_fresh.pt"), weights_only=False)
    assert "reference" in blob["source"]
    c = blob["case"]
    assert c["data"].shape == (1500, 24) and c["k"] == 32
    got = io.kmeans(c["data"], c["k"], c["niters"], c["seed"], c["max_points_per_centroid"])
    assert torch.equal(got, c["centroids"]), float((got - c["centroids"]).abs().max())
