"""The fp64 intervals of tests/util.py are not vacuous.

The oracle's own fp16 arithmetic (ATen CPU: fp32-accumulated half matmul, fp16 norm, IEEE division, fp16 max, fp32
sum) must lie inside them, and each of the small errors a kernel could make must land outside them: a dropped last
token, a column maximum two fp16 ulps off, a padded query column summed into an empty document's score.
"""

from __future__ import annotations

import pytest
import torch

from util import (PAD_SENTINEL, build_oracle_index, centroid_score_bounds, f16_step, interval_report, make_docs,
                  make_queries, maxsim_bounds, normalise_like_the_kernels, oracle_exact_scores, round_down_f16,
                  round_up_f16, token_norm_bounds)

from oracle import plaid_oracle as po


@pytest.fixture(scope="module")
def case():
    docs = make_docs(40, 5, 40, seed=21)
    oidx, _ = build_oracle_index(docs, kmeans_niters=2)
    lens = oidx.doc_lengths.clone()
    lens[6] += lens[5]
    lens[5] = 0  # document 5 has no tokens
    oidx = po.OracleIndex(oidx.nbits, oidx.centroids, oidx.bucket_weights, oidx.ivf, oidx.ivf_lengths, oidx.doc_codes,
                          oidx.doc_residuals, lens)
    T = int(oidx.doc_offsets[-1])
    e16 = po.decode_unnormalised(oidx.doc_residuals[:T], oidx.bucket_weights, oidx.byte_reversed_bits_map,
                                 oidx.bucket_weight_indices_lookup, oidx.doc_codes[:T], oidx.centroids, oidx.dim,
                                 oidx.nbits)
    norms = torch.linalg.vector_norm(e16, ord=2.0, dim=-1)  # fp16, as the reference computes it
    ehat = normalise_like_the_kernels(e16, norms)
    return oidx, e16, norms, ehat


def _inside(s: float, bound: tuple[float, float]) -> bool:
    return bound[0] <= s <= bound[1]


def _planted_query(ehat, row: int, Q: int, seed: int, dim: int = 128) -> torch.Tensor:
    """Q query tokens; token 0 is the (noisy) copy of token `row`, so that token holds column 0's maximum."""
    q = make_queries(1, Q, dim=dim, seed=seed)[0]
    q[0] = torch.nn.functional.normalize(ehat[row].float() + 0.02 * torch.randn(dim), dim=0)
    return q.half()


def test_rounding_helpers():
    x = torch.tensor([1.0, 1.0 + 2**-12, -1.0 - 2**-12, 0.0, 65504.0, 1e-9, -1e-9], dtype=torch.float64)
    lo, hi = round_down_f16(x), round_up_f16(x)
    assert lo.tolist() == [1.0, 1.0, -1.0 - 2**-10, 0.0, 65504.0, 0.0, -(2.0**-24)]
    assert hi.tolist() == [1.0, 1.0 + 2**-10, -1.0, 0.0, 65504.0, 2.0**-24, 0.0]
    h = torch.tensor([1.0, -1.0, 0.0], dtype=torch.float16)
    assert f16_step(h, 1).tolist() == [1.0 + 2**-10, -1.0 + 2**-11, 2.0**-24]
    assert f16_step(h, -1).tolist() == [1.0 - 2**-11, -1.0 - 2**-10, -(2.0**-24)]


def test_oracle_fp16_arithmetic_is_inside_the_bounds(case):
    oidx, e16, norms, ehat = case
    q16 = make_queries(2, 32, seed=5).half()
    for b in range(2):
        S = oidx.centroids.matmul(q16[b].t())  # search.rs:491 on ATen's CPU half matmul
        lo, hi, x, g = centroid_score_bounds(oidx.centroids, q16[b])
        assert not interval_report(S, lo, hi, x, g)
    lo, hi = token_norm_bounds(e16)
    assert bool(((norms >= lo) & (norms <= hi)).all())
    docs = list(range(oidx.doc_lengths.shape[0]))
    offs, lens = oidx.doc_offsets[:-1].tolist(), oidx.doc_lengths.tolist()
    for b in range(2):
        got = oracle_exact_scores(oidx, q16[b].float(), docs)
        bounds = maxsim_bounds(ehat, offs, lens, q16[b])
        for d in docs:
            assert _inside(float(got[d]), bounds[d]), (d, float(got[d]), bounds[d])
    assert bounds[5] == (32 * PAD_SENTINEL, 32 * PAD_SENTINEL)


def _score(ehat_rows: torch.Tensor, q16: torch.Tensor, extra_cols: int = 0) -> float:
    """The oracle's MaxSim of one document given its normalised rows (colbert_score_reduce), optionally over
    `extra_cols` more query columns of zeros (the padded columns of a kernel's query tile)."""
    if extra_cols:
        q16 = torch.cat([q16, torch.zeros(extra_cols, q16.shape[1], dtype=q16.dtype)])
    n = ehat_rows.shape[0]
    ts = ehat_rows.unsqueeze(0).matmul(q16.t())  # [1, n, Q]
    mask = torch.ones(1, n, dtype=torch.bool)
    if n == 0:
        ts = torch.zeros(1, 1, q16.shape[0], dtype=torch.float16)
        mask = torch.zeros(1, 1, dtype=torch.bool)
    return float(po.colbert_score_reduce(ts, mask)[0])


@pytest.mark.parametrize("Q", [1, 32, 256])
def test_dropping_the_last_token_is_caught(case, Q):
    oidx, e16, norms, ehat = case
    offs, lens = oidx.doc_offsets[:-1].tolist(), oidx.doc_lengths.tolist()
    for d in (0, 7, 12):
        o, n = offs[d], lens[d]
        q16 = _planted_query(ehat, o + n - 1, Q, seed=d)
        bound = maxsim_bounds(ehat, [o], [n], q16)[0]
        assert _inside(_score(ehat[o : o + n], q16), bound)
        assert not _inside(_score(ehat[o : o + n - 1], q16), bound), f"doc {d}: a dropped last token passes"


def test_a_column_maximum_two_ulps_off_is_caught(case):
    """One query token: the score is the column maximum itself, so two fp16 ulps are outside the interval (with many
    columns the interval of the sum is as wide as the sum of the per-column roundings; the GPU tests plant maxima so
    that an error moves a score by far more)."""
    oidx, e16, norms, ehat = case
    offs, lens = oidx.doc_offsets[:-1].tolist(), oidx.doc_lengths.tolist()
    for d in (0, 3, 9):
        o, n = offs[d], lens[d]
        q16 = _planted_query(ehat, o + n // 2, 1, seed=100 + d)
        bound = maxsim_bounds(ehat, [o], [n], q16)[0]
        ts = ehat[o : o + n].matmul(q16.t())[:, 0]
        m = ts.max().reshape(1)
        assert _inside(float(m.float()), bound)
        for direction in (1, -1):
            off = f16_step(f16_step(m, direction), direction)
            assert not _inside(float(off.float()), bound), f"doc {d}: a maximum 2 ulps off passes"


def test_a_padded_column_in_an_empty_document_is_caught(case):
    oidx, e16, norms, ehat = case
    q16 = make_queries(1, 20, seed=3)[0].half()
    bound = maxsim_bounds(ehat, [int(oidx.doc_offsets[5])], [0], q16)[0]
    empty = ehat[:0]
    assert _inside(_score(empty, q16), bound)
    assert not _inside(_score(empty, q16, extra_cols=1), bound)
