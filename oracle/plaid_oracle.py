"""CPU oracle for the fast-plaid search hot path.  TEST INFRASTRUCTURE ONLY.

This module is the parity checker for the B200 engine.  Only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl reference``
legs may import it.  Nothing under ``fast_plaid_b200/`` imports it, and the product
path never falls back to it.

What it is
----------
An op-for-op PyTorch-CPU restatement of the reference's Rust search pipeline.  The
reference (lightonai/fast-plaid v1.4.6 @ 87f96f6) has no kernels of its own: every
numeric operation in ``rust/search/search.rs`` is a libtorch ATen call made through
``tch = "0.20.0"`` (``Cargo.toml:15``; there is no ``Cargo.lock``), and the reference's
CI runs against ``torch==2.11.0`` (``.github/workflows/tests.yaml:40``) -- the very
ATen build importable in this image.  Issuing the same ATen op sequence from Python
therefore executes the same CPU kernels with the same fp16 rounding points.

PARITY UNPINNED: the reference cannot be built here (Rust/maturin/cargo absent, no
wheel, no network) and its own tests (``tests/test.py``) hold no golden vectors or
known-answer values for this path (all inputs are unseeded ``torch.randn``).  The only
numeric relations the reference pins -- ``search`` vs ``search_token_scores`` ids equal
and |dscore| < 1e-3 (``tests/test.py:143-173``) and manual ``max(dim=1).sum()`` within
0.1 of the returned score (``tests/test.py:175-197``) -- are re-checked against this
oracle in ``tests/test_oracle.py``.  Golden fixtures under ``tests/golden/`` are
minted by this oracle (``tests/golden/make_golden.py``), not by the reference.

Two tie modes
-------------
``ties="torch"``      exactly the reference op sequence: ``topk``/``sort`` resolve ties
                      however ATen's CPU kernels do (implementation-defined; probed
                      here: neither ``topk`` nor non-stable ``sort`` keeps index order).
``ties="canonical"``  identical arithmetic, but every implementation-defined choice is
                      resolved by one stated rule: larger value first, then smaller
                      index (centroid id / doc id).  This is the rule the CUDA engine
                      implements; ``tests/test_oracle.py`` shows the two modes agree
                      wherever the reference's result is well defined.
"""

from __future__ import annotations

import dataclasses
from typing import Any

import torch

# --------------------------------------------------------------------------------------
# Index container (mirrors LoadedIndex / ResidualCodec / StridedTensor state,
# rust/search/load.rs:50-56, rust/utils/residual_codec.rs:15-34, rust/search/tensor.rs:132-147)
# --------------------------------------------------------------------------------------


@dataclasses.dataclass
class OracleIndex:
    nbits: int
    centroids: torch.Tensor  # f16 [K, D]              load.rs:145-152 casts to Half
    bucket_weights: torch.Tensor  # f16 [2**nbits]      load.rs:150
    ivf: torch.Tensor | None  # i64 [n_ivf]             load.rs:158-164
    ivf_lengths: torch.Tensor | None  # i64 [K]         tensor.rs:211 (Int -> Int64)
    doc_codes: torch.Tensor  # i64 [E]
    doc_residuals: torch.Tensor  # u8 [E, D*nbits/8]
    doc_lengths: torch.Tensor  # i64 [N]
    # derived
    byte_reversed_bits_map: torch.Tensor = None  # u8 [256]
    bucket_weight_indices_lookup: torch.Tensor = None  # i64 [256, 8/nbits]
    ivf_offsets: torch.Tensor = None  # i64 [K+1]
    doc_offsets: torch.Tensor = None  # i64 [N+1]

    def __post_init__(self) -> None:
        self.centroids = self.centroids.to(torch.float16)
        self.bucket_weights = self.bucket_weights.to(torch.float16)
        self.doc_codes = self.doc_codes.to(torch.int64)
        self.doc_lengths = self.doc_lengths.to(torch.int64)
        self.byte_reversed_bits_map, self.bucket_weight_indices_lookup = codec_luts(self.nbits)
        z = torch.zeros(1, dtype=torch.int64)
        self.doc_offsets = torch.cat([z, self.doc_lengths.cumsum(0)])
        if self.ivf is not None:
            self.ivf = self.ivf.to(torch.int64)
            self.ivf_lengths = self.ivf_lengths.to(torch.int64)
            self.ivf_offsets = torch.cat([z, self.ivf_lengths.cumsum(0)])

    @property
    def dim(self) -> int:
        return int(self.centroids.shape[1])


def codec_luts(nbits: int) -> tuple[torch.Tensor, torch.Tensor]:
    """The two 256-entry tables of ``ResidualCodec::load`` (residual_codec.rs:83-140)."""
    mask = (1 << nbits) - 1
    rev = [0] * 256
    for i in range(256):
        out = 0
        pos = 8
        while pos >= nbits:  # residual_codec.rs:91
            segment = (i >> (pos - nbits)) & mask
            rev_segment = 0
            for k in range(nbits):  # residual_codec.rs:95-99
                if segment & (1 << k):
                    rev_segment |= 1 << (nbits - 1 - k)
            out |= rev_segment
            if pos > nbits:
                out <<= nbits
            pos -= nbits
        rev[i] = out & 0xFF
    keys_per_byte = 8 // nbits
    table = []
    for byte_val in range(256):  # residual_codec.rs:124-130
        for k in reversed(range(keys_per_byte)):
            table.append((byte_val >> (k * nbits)) & mask)
    return (
        torch.tensor(rev, dtype=torch.uint8),
        torch.tensor(table, dtype=torch.int64).reshape(256, keys_per_byte),
    )


# --------------------------------------------------------------------------------------
# StridedTensor::lookup  (rust/search/tensor.rs:299-355)
# The strided-window + boolean-mask compaction returns, in index order, the concatenation
# of rows [off[i], off[i]+len[i]) of the flat data tensor.  That is what is restated here;
# the choice of window stride (tensor.rs:322-327, randint-sampled quantiles :163-165)
# affects only how many padding rows are read and then masked away, never the result.
# --------------------------------------------------------------------------------------


def ragged_lookup(
    data: torch.Tensor, offsets: torch.Tensor, lengths: torch.Tensor, indices: torch.Tensor
) -> tuple[torch.Tensor, torch.Tensor]:
    indices = indices.to(torch.int64)
    if indices.numel() == 0:  # tensor.rs:304-311
        return data.new_empty((0,) + tuple(data.shape[1:])), lengths.new_empty((0,))
    sel_len = lengths.index_select(0, indices)  # tensor.rs:313
    sel_off = offsets.index_select(0, indices)  # tensor.rs:314
    total = int(sel_len.sum())
    if total == 0:
        return data.new_empty((0,) + tuple(data.shape[1:])), sel_len
    starts = sel_len.cumsum(0) - sel_len
    within = torch.arange(total, dtype=torch.int64) - torch.repeat_interleave(starts, sel_len)
    rows = torch.repeat_interleave(sel_off, sel_len) + within
    return data.index_select(0, rows), sel_len


# --------------------------------------------------------------------------------------
# direct_pad_sequences  (rust/search/padding.rs:61-109)
# --------------------------------------------------------------------------------------


def direct_pad_sequences(
    sequences: torch.Tensor, lengths: torch.Tensor, pad_value: float
) -> tuple[torch.Tensor, torch.Tensor]:
    if lengths.numel() == 0:  # padding.rs:67-72
        return (
            sequences.new_empty((0, 0, sequences.shape[1])),
            torch.empty((0, 0), dtype=torch.bool),
        )
    batch = lengths.shape[0]
    feat = sequences.shape[1]
    max_len = int(lengths.max())  # padding.rs:77-78
    padded = torch.full((batch, max_len, feat), pad_value, dtype=sequences.dtype)  # :80-87
    mask = torch.arange(max_len, dtype=torch.int64).unsqueeze(0) < lengths.unsqueeze(-1)  # :90-93
    nz = mask.nonzero()  # :96
    padded.index_put_((nz[:, 0], nz[:, 1]), sequences, accumulate=False)  # :102-106
    return padded, mask


# --------------------------------------------------------------------------------------
# colbert_score_reduce  (rust/search/search.rs:385-402)
# --------------------------------------------------------------------------------------


def colbert_score_reduce(token_scores: torch.Tensor, attention_mask: torch.Tensor) -> torch.Tensor:
    expanded = attention_mask.unsqueeze(-1).expand(token_scores.shape)  # :389
    padding = expanded.logical_not()  # :392
    masked = token_scores.masked_fill(padding, -9999.0)  # :395  (fp16: -9999 -> -10000)
    max_per_token = masked.max(dim=1).values  # :398
    return max_per_token.sum(dim=-1, dtype=torch.float32)  # :401  (Kind::Float)


# --------------------------------------------------------------------------------------
# decompress_residuals  (rust/search/search.rs:53-107)
# --------------------------------------------------------------------------------------


def decompress_residuals(
    packed_residuals: torch.Tensor,
    bucket_weights: torch.Tensor,
    byte_reversed_bits_map: torch.Tensor,
    bucket_weight_indices_lookup: torch.Tensor,
    codes: torch.Tensor,
    centroids: torch.Tensor,
    embedding_dimension: int,
    nbits: int,
) -> torch.Tensor:
    emb = decode_unnormalised(packed_residuals, bucket_weights, byte_reversed_bits_map, bucket_weight_indices_lookup,
                              codes, centroids, embedding_dimension, nbits)
    norms = torch.linalg.vector_norm(emb, ord=2.0, dim=-1, keepdim=True).clamp_min(1e-12)  # :101-103
    return emb / norms  # :105


def decode_unnormalised(
    packed_residuals: torch.Tensor,
    bucket_weights: torch.Tensor,
    byte_reversed_bits_map: torch.Tensor,
    bucket_weight_indices_lookup: torch.Tensor,
    codes: torch.Tensor,
    centroids: torch.Tensor,
    embedding_dimension: int,
    nbits: int,
) -> torch.Tensor:
    """The decoded tokens before normalisation, e = fp16(w + c) (search.rs:66-99)."""
    n = codes.shape[0]
    packed_dim = (embedding_dimension * nbits) // 8  # :66
    per_byte = 8 // nbits  # :67
    retrieved = centroids.index_select(0, codes)  # :70
    reshaped_centroids = retrieved.view(n, packed_dim, per_byte)  # :71-72
    flat_idx = packed_residuals.flatten().to(torch.int32)  # :75
    flat_rev = byte_reversed_bits_map.index_select(0, flat_idx).to(torch.uint8)  # :76-78
    flat_sel = bucket_weight_indices_lookup.index_select(0, flat_rev.to(torch.int32)).to(
        torch.uint8
    )  # :83-85
    flat_bucket_idx = flat_sel.view(n, packed_dim, per_byte).flatten()  # :86-90
    gathered = bucket_weights.index_select(0, flat_bucket_idx.to(torch.int32))  # :91-92
    reshaped_w = gathered.view(n, packed_dim, per_byte)  # :93-94
    summed = reshaped_w + reshaped_centroids  # :97
    return summed.view(n, embedding_dimension)  # :98-99


# --------------------------------------------------------------------------------------
# Canonical tie rule helpers
# --------------------------------------------------------------------------------------


def _topk_indices(values: torch.Tensor, k: int, ties: str, sorted_: bool) -> torch.Tensor:
    """Indices of the k largest entries of a 1-D tensor."""
    if ties == "torch":
        return values.topk(k, 0, True, sorted_).indices
    # canonical: value desc, index asc  (stable descending sort keeps index order in ties)
    order = torch.sort(values.float(), descending=True, stable=True).indices
    return order[:k]


def _topk_rows_per_column(scores: torch.Tensor, k: int, ties: str) -> torch.Tensor:
    """[K, Q] -> [k, Q] row indices of the k largest per column (search.rs:520-527)."""
    if ties == "torch":
        if k == 1:
            return scores.argmax(0, keepdim=True)
        return scores.topk(k, 0, True, False).indices
    order = torch.sort(scores.float(), dim=0, descending=True, stable=True).indices
    return order[:k]


# --------------------------------------------------------------------------------------
# search  (rust/search/search.rs:471-696)
# --------------------------------------------------------------------------------------


def search_one(
    query: torch.Tensor,
    index: OracleIndex,
    n_ivf_probe: int = 8,
    batch_size: int = 2000,
    n_full_scores: int = 4096,
    top_k: int = 10,
    subset: torch.Tensor | None = None,
    ties: str = "torch",
    return_stages: bool = False,
    inject: dict[str, torch.Tensor] | None = None,
) -> Any:
    """One query [Q, D] (any float dtype; cast to fp16 as fast_plaid.py:241 does).

    ``inject`` lets a test substitute a stage output computed elsewhere (e.g. the GPU's
    centroid-score table ``S``) to check that everything downstream of it is bit-exact;
    ``inject["subset_centroids"]`` replaces the centroid set derived from the subset documents
    (the document-sharded engine uses the union over the shards, tests/test_sharding.py).
    Returns (passage_ids: list[int], scores: list[float]) or, with ``return_stages``, a
    dict that also holds every intermediate.
    """
    inject = inject or {}
    st: dict[str, Any] = {}
    q = query.to(torch.float16)  # fast_plaid.py:241
    d = index.dim
    q_unsq = q.unsqueeze(0)  # :488

    S = inject.get("S")
    if S is None:
        S = index.centroids.matmul(q.transpose(0, 1))  # :491   [K, Q] fp16
    st["S"] = S

    if index.ivf is None:
        raise ValueError(
            "This index was built with compress_only=True and does not support search. "
            "Rebuild with compress_only=False to enable search."
        )  # :227-232

    if subset is not None:  # :494-517
        subset = subset.to(torch.int64)
        subset_codes, _ = ragged_lookup(index.doc_codes, index.doc_offsets, index.doc_lengths, subset)
        uniq_c = torch.unique(subset_codes.flatten(), sorted=True)
        st["subset_centroids"] = uniq_c
        if "subset_centroids" in inject:
            uniq_c = inject["subset_centroids"].to(torch.int64)
        if uniq_c.numel() == 0:
            flat_cells = torch.empty(0, dtype=torch.int64)
        else:
            sub_scores = S.index_select(0, uniq_c)
            actual_k = min(n_ivf_probe, uniq_c.shape[0])
            local = _topk_rows_per_column(sub_scores, actual_k, ties)
            flat_cells = uniq_c.index_select(0, local.flatten())
    else:  # :519-529
        cells = _topk_rows_per_column(S, n_ivf_probe, ties)  # [n_probe, Q]
        flat_cells = cells.permute(1, 0).flatten().contiguous()
    st["probe_cells"] = flat_cells

    uniq_cells = torch.unique(flat_cells, sorted=True)  # :531-532
    st["cells"] = uniq_cells

    pids_ivf, _ = ragged_lookup(index.ivf, index.ivf_offsets, index.ivf_lengths, uniq_cells)  # :535
    sorted_pids = pids_ivf.sort(0, False).values  # :538
    uniq_pids = torch.unique_consecutive(sorted_pids)  # :540-541

    if subset is not None:  # :544-547, :430-439, :407-427
        if subset.numel() == 0 or uniq_pids.numel() == 0:
            uniq_pids = torch.empty(0, dtype=torch.int64)
        else:
            us = torch.unique_consecutive(subset.sort(0, False).values)
            cat = torch.cat([uniq_pids, us]).sort(0, False).values
            if cat.shape[0] < 2:
                uniq_pids = torch.empty(0, dtype=torch.int64)
            else:
                dup = cat[:-1] == cat[1:]
                uniq_pids = cat[1:][dup]
    st["candidates"] = uniq_pids

    if uniq_pids.numel() == 0:  # :549-551
        return _finish([], [], st, return_stages)

    chunks = []
    total = uniq_pids.shape[0]
    for start in range(0, total, batch_size):  # :558-586
        batch_pids = uniq_pids[start : start + batch_size]
        codes, lens = ragged_lookup(index.doc_codes, index.doc_offsets, index.doc_lengths, batch_pids)
        if codes.numel() == 0:  # :570-576
            chunks.append(torch.zeros(batch_pids.shape[0], dtype=torch.float32))
            continue
        gathered = S.index_select(0, codes)  # :578
        padded, mask = direct_pad_sequences(gathered, lens, 0.0)  # :580-581
        chunks.append(colbert_score_reduce(padded, mask))  # :583
    approx = torch.cat(chunks, 0)  # :588-592
    st["approx"] = approx
    if "approx" in inject:  # tests: prune on approximate scores computed elsewhere (same candidate order)
        approx = inject["approx"].to(torch.float32)

    rerank = uniq_pids
    if n_full_scores < approx.shape[0]:  # :605-611
        top_idx = _topk_indices(approx, n_full_scores, ties, True)
        rerank = rerank.index_select(0, top_idx)
        approx = approx.index_select(0, top_idx)
    n_dec = max(n_full_scores // 4, 1)  # :614
    if n_dec < approx.shape[0]:  # :615-619
        top_idx = _topk_indices(approx, n_dec, ties, True)
        rerank = rerank.index_select(0, top_idx)
    st["rerank"] = rerank

    if rerank.numel() == 0:  # :621-623
        return _finish([], [], st, return_stages)

    final_codes, final_lens = ragged_lookup(
        index.doc_codes, index.doc_offsets, index.doc_lengths, rerank
    )  # :626-627
    final_res, _ = ragged_lookup(index.doc_residuals, index.doc_offsets, index.doc_lengths, rerank)  # :629
    emb = decompress_residuals(
        final_res,
        index.bucket_weights,
        index.byte_reversed_bits_map,
        index.bucket_weight_indices_lookup,
        final_codes,
        index.centroids,
        d,
        index.nbits,
    )  # :640-649
    if return_stages:
        st["embeddings"] = emb
        st["rerank_lengths"] = final_lens
    padded_emb, mask = direct_pad_sequences(emb, final_lens, 0.0)  # :651-652
    ts = inject.get("token_scores")
    if ts is None:
        ts = padded_emb.matmul(q_unsq.transpose(-2, -1))  # :654-655   [R, L, Q] fp16
    exact = colbert_score_reduce(ts, mask)  # :656
    st["exact"] = exact
    if return_stages:
        st["token_scores"] = ts

    if ties == "torch":
        sorted_scores, order = exact.sort(0, True)  # :659
    else:
        # canonical: score desc, doc id asc
        by_id = torch.sort(rerank, stable=True).indices
        o2 = torch.sort(exact.index_select(0, by_id), descending=True, stable=True).indices
        order = by_id.index_select(0, o2)
        sorted_scores = exact.index_select(0, order)
    sorted_pids = rerank.index_select(0, order)  # :661
    n_out = min(top_k, sorted_pids.shape[0])  # :666
    st["order"] = order
    ids = sorted_pids[:n_out].tolist()
    sc = sorted_scores[:n_out].tolist()
    if return_stages:
        st["token_matrices"] = [
            ts[int(order[i])][: int(final_lens[int(order[i])])].transpose(0, 1) for i in range(n_out)
        ]  # :668-686
    return _finish(ids, sc, st, return_stages)


def _finish(ids, sc, st, return_stages):
    if return_stages:
        st["ids"] = ids
        st["scores"] = sc
        return st
    return ids, sc


def search_many(
    queries: torch.Tensor,
    index: OracleIndex,
    n_ivf_probe: int = 8,
    batch_size: int = 2000,
    n_full_scores: int = 4096,
    top_k: int = 10,
    subset: list[list[int]] | None = None,
    ties: str = "torch",
) -> list[list[tuple[int, float]]]:
    """search_many + the re-zip of search_on_device (search.rs:219-288, fast_plaid.py:247-253)."""
    if queries.dim() != 3:
        raise ValueError(f"Expected a 3D tensor for queries, but got shape {list(queries.shape)}")
    out = []
    with torch.no_grad():
        for i in range(queries.shape[0]):
            sub = None
            if subset is not None and i < len(subset):
                sub = torch.tensor(subset[i], dtype=torch.int64)
            try:
                ids, sc = search_one(
                    queries[i], index, n_ivf_probe, batch_size, n_full_scores, top_k, sub, ties
                )
            except ValueError:
                raise
            except Exception:  # search.rs:268 .unwrap_or_default()
                ids, sc = [], []
            out.append(list(zip(ids, sc)))
    return out
