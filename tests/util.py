"""Shared helpers for the parity tests (seeded synthetic indexes, tolerant comparisons)."""

from __future__ import annotations

import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import index_oracle, plaid_oracle  # noqa: E402


def make_docs(n_docs: int, min_len: int, max_len: int, dim: int = 128, seed: int = 1234,
              normalize: bool = True) -> list[torch.Tensor]:
    g = torch.Generator().manual_seed(seed)
    lens = torch.randint(min_len, max_len + 1, (n_docs,), generator=g)
    docs = []
    for ln in lens.tolist():
        x = torch.randn(ln, dim, generator=g)
        docs.append(torch.nn.functional.normalize(x, dim=-1) if normalize else x)
    return docs


def make_queries(B: int, Q: int, dim: int = 128, seed: int = 4321, docs: list[torch.Tensor] | None = None,
                 noise: float = 0.2) -> torch.Tensor:
    """Random unit queries, or (with `docs`) noisy copies of document tokens -- the second
    kind gives well separated scores like real retrieval (SURVEY.md 8d)."""
    g = torch.Generator().manual_seed(seed)
    if docs is None:
        return torch.nn.functional.normalize(torch.randn(B, Q, dim, generator=g), dim=-1)
    out = []
    for _ in range(B):
        d = docs[int(torch.randint(0, len(docs), (1,), generator=g))]
        rows = torch.randint(0, d.shape[0], (Q,), generator=g)
        x = d[rows].float() + noise * torch.randn(Q, dim, generator=g)
        out.append(torch.nn.functional.normalize(x, dim=-1))
    return torch.stack(out)


def build_oracle_index(docs, nbits: int = 4, seed: int = 42, kmeans_niters: int = 4):
    cent = index_oracle.compute_centroids(docs, kmeans_niters, seed)
    idx, extra = index_oracle.build_index(docs, cent, nbits=nbits, seed=seed)
    return idx, extra


def to_index_tensors(idx: plaid_oracle.OracleIndex):
    from fast_plaid_b200.engine import IndexTensors

    return IndexTensors(
        nbits=idx.nbits,
        centroids=idx.centroids,
        bucket_weights=idx.bucket_weights,
        doc_lengths=idx.doc_lengths,
        doc_codes=idx.doc_codes,
        doc_residuals=idx.doc_residuals,
        ivf=idx.ivf,
        ivf_lengths=idx.ivf_lengths,
    )


def fp16_ulp_diff(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """Distance in representable fp16 steps between two fp16 tensors."""
    def key(x):
        i = x.contiguous().view(torch.int16).to(torch.int32)
        return torch.where(i < 0, -(i & 0x7FFF), i)
    return (key(a.half()) - key(b.half())).abs()


def oracle_exact_scores(oidx, query: torch.Tensor, doc_ids: list[int]) -> torch.Tensor:
    """Reference exact MaxSim score (search.rs:626-656) of arbitrary documents."""
    sel = torch.tensor(doc_ids, dtype=torch.int64)
    codes, lens = plaid_oracle.ragged_lookup(oidx.doc_codes, oidx.doc_offsets, oidx.doc_lengths, sel)
    res, _ = plaid_oracle.ragged_lookup(oidx.doc_residuals, oidx.doc_offsets, oidx.doc_lengths, sel)
    emb = plaid_oracle.decompress_residuals(res, oidx.bucket_weights, oidx.byte_reversed_bits_map,
                                            oidx.bucket_weight_indices_lookup, codes, oidx.centroids, oidx.dim,
                                            oidx.nbits)
    padded, mask = plaid_oracle.direct_pad_sequences(emb, lens, 0.0)
    ts = padded.matmul(query.half().unsqueeze(0).transpose(-2, -1))
    return plaid_oracle.colbert_score_reduce(ts, mask)


def oracle_token_matrix(oidx, query: torch.Tensor, doc_id: int) -> torch.Tensor:
    """Reference token-score matrix (search.rs:651-655 then :668-686) of one document: fp16 [Q, len]."""
    sel = torch.tensor([doc_id], dtype=torch.int64)
    codes, lens = plaid_oracle.ragged_lookup(oidx.doc_codes, oidx.doc_offsets, oidx.doc_lengths, sel)
    res, _ = plaid_oracle.ragged_lookup(oidx.doc_residuals, oidx.doc_offsets, oidx.doc_lengths, sel)
    emb = plaid_oracle.decompress_residuals(res, oidx.bucket_weights, oidx.byte_reversed_bits_map,
                                            oidx.bucket_weight_indices_lookup, codes, oidx.centroids, oidx.dim,
                                            oidx.nbits)
    padded, _ = plaid_oracle.direct_pad_sequences(emb, lens, 0.0)
    ts = padded.matmul(query.half().unsqueeze(0).transpose(-2, -1))  # [1, len, Q]
    return ts[0, : int(lens[0])].transpose(0, 1).contiguous()


def ranking_consistent(gpu_ids, gpu_scores, ref_score_of: dict, tol: float, fallback=None) -> tuple[bool, str]:
    """The GPU ranking must be a valid ranking of the reference scores up to `tol`:
    every returned doc has (nearly) the reference score, and no doc is ranked above another
    whose reference score is larger by more than tol.  A doc the reference run did not
    re-rank (possible only through a tie at a topk boundary) is scored through `fallback`."""
    prev = None
    for i, (d, s) in enumerate(zip(gpu_ids, gpu_scores)):
        if d not in ref_score_of:
            if fallback is None:
                return False, f"rank {i}: doc {d} was not scored by the reference"
            ref_score_of[d] = fallback(d)
        r = ref_score_of[d]
        if abs(r - s) > tol * max(1.0, abs(r)):
            return False, f"rank {i}: doc {d} score {s} vs reference {r}"
        if prev is not None and r > prev + tol * max(1.0, abs(r)):
            return False, f"rank {i}: doc {d} (ref {r}) ranked below a doc with ref {prev}"
        prev = r
    return True, ""


# ---- fp64 references with stated error bounds (DESIGN.md "Parity contract") -----------------------------------
# Every rounding step of the search arithmetic is one IEEE operation, so each fp16 result the kernels produce must lie
# in an interval around the exact (fp64) value: the fp32 error bound of the accumulation, widened outward to fp16.
U32 = 2.0 ** -24  # unit roundoff of fp32
# a dot product of at most 128 fp16 x fp16 products (each exact in fp32) accumulated in fp32: |err| <= 128 u sum|c q|
DOT_TERMS = 128
PAD_SENTINEL = -10000.0  # fp16(-9999), the score of a query token against a document without tokens


def f16_step(h: torch.Tensor, direction: int) -> torch.Tensor:
    """The fp16 neighbour of every entry of `h` (fp16) towards +inf (direction 1) or -inf (-1)."""
    i = h.contiguous().view(torch.int16).to(torch.int32)
    key = torch.where(i < 0, -(i & 0x7FFF), i) + direction  # order-preserving integer line, -0 and +0 both 0
    bits = torch.where(key < 0, (-key) | 0x8000, key)
    return torch.where(bits >= 0x8000, bits - 0x10000, bits).to(torch.int16).view(torch.float16)


def round_down_f16(x: torch.Tensor) -> torch.Tensor:
    """Largest fp16 <= x (x fp64)."""
    h = x.half()
    return torch.where(h.double() > x, f16_step(h, -1), h)


def round_up_f16(x: torch.Tensor) -> torch.Tensor:
    """Smallest fp16 >= x (x fp64)."""
    h = x.half()
    return torch.where(h.double() < x, f16_step(h, 1), h)


def dot_fp64(a16: torch.Tensor, b16: torch.Tensor) -> tuple[torch.Tensor, torch.Tensor]:
    """x = a . b^T in fp64 and gamma = 128 u sum|a b|, its fp32-accumulation bound ([n, D] x [m, D] -> [n, m])."""
    a, b = a16.double(), b16.double()
    return a @ b.T, DOT_TERMS * U32 * (a.abs() @ b.abs().T)


def centroid_score_bounds(centroids16: torch.Tensor, q16: torch.Tensor) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """fp16 [K, Q] interval [RD16(x - gamma), RU16(x + gamma)] every S[k, q] must lie in; also returns x and gamma."""
    x, g = dot_fp64(centroids16, q16)
    return round_down_f16(x - g), round_up_f16(x + g), x, g


def interval_report(got: torch.Tensor, lo: torch.Tensor, hi: torch.Tensor, x: torch.Tensor, g: torch.Tensor) -> str:
    """'' when lo <= got <= hi everywhere, else the count and the worst |got - x| / gamma among the violations."""
    gd = got.double()
    bad = (gd < lo.double()) | (gd > hi.double()) | torch.isnan(gd)
    if not bool(bad.any()):
        return ""
    ratio = ((gd - x).abs() / g.clamp_min(1e-300))[bad]
    return f"{int(bad.sum())} of {bad.numel()} entries outside the fp64 interval, worst |err| / gamma = {float(ratio.max()):.3g}"


def token_norm_bounds(e16: torch.Tensor) -> tuple[torch.Tensor, torch.Tensor]:
    """fp16 interval of fp16(sqrt(sum_fp32 e^2)) per row of e (fp16 [n, D]): the fp32 sum of the D exact squares is
    within 128 u of the fp64 one, the square root adds one rounding."""
    ss = (e16.double() ** 2).sum(-1)
    lo = torch.sqrt(ss * (1 - DOT_TERMS * U32)) * (1 - U32)
    hi = torch.sqrt(ss * (1 + DOT_TERMS * U32)) * (1 + U32)
    return round_down_f16(lo), round_up_f16(hi)


def normalise_like_the_kernels(e16: torch.Tensor, norms16: torch.Tensor) -> torch.Tensor:
    """e_hat = fp16(fp32(e) / fp32(n)): one IEEE division (exact on the CPU), one rounding."""
    return (e16.float() / norms16.float().unsqueeze(-1)).half()


def maxsim_bounds(ehat16: torch.Tensor, offsets: list[int], lengths: list[int], q16: torch.Tensor,
                  x: torch.Tensor | None = None, g: torch.Tensor | None = None) -> list[tuple[float, float]]:
    """Interval [lo, hi] of the exact MaxSim score of each document (rows offsets[i] .. + lengths[i] of ehat16)
    against the query q16 [Q, D]:  lo_q = RD16(max_t(x_tq - gamma_tq)),  hi_q = RU16(max_t(x_tq + gamma_tq)),
    score in [sum lo_q - eps, sum hi_q + eps] with eps = Q u sum max(|lo_q|, |hi_q|) for the fp32 sum over q.
    A document without tokens scores exactly Q * -10000 (lo == hi).  `x` / `g` may hold dot_fp64(ehat16, q16)."""
    Q = q16.shape[0]
    if x is None:
        x, g = dot_fp64(ehat16, q16)
    out = []
    for o, n in zip(offsets, lengths):
        if n == 0:
            out.append((Q * PAD_SENTINEL, Q * PAD_SENTINEL))
            continue
        lo_q = round_down_f16((x[o : o + n] - g[o : o + n]).max(0).values).double()
        hi_q = round_up_f16((x[o : o + n] + g[o : o + n]).max(0).values).double()
        eps = Q * U32 * float(torch.maximum(lo_q.abs(), hi_q.abs()).sum())
        out.append((float(lo_q.sum()) - eps, float(hi_q.sum()) + eps))
    return out


def merge_records_host(records: list[tuple[float, float, int]], R: int, top_k: int) -> list[tuple[int, float]]:
    """Host statement of the sharded merge rule (k6_merge_kernel): keep the R best by
    (approx desc, doc id asc), order them by (exact desc, doc id asc), emit top_k."""
    keep = sorted(records, key=lambda r: (-r[0], r[2]))[:R]
    keep.sort(key=lambda r: (-r[1], r[2]))
    return [(r[2], r[1]) for r in keep[:top_k]]


def shard_records_oracle(shard_index, base: int, query: torch.Tensor, n_probe: int, n_full: int):
    """What fpb_search_shard emits for one query, computed with the oracle on a shard."""
    st = plaid_oracle.search_one(query, shard_index, n_probe, 2000, n_full, 10**9, ties="canonical",
                                 return_stages=True)
    if len(st.get("ids", [])) == 0 and "rerank" not in st:
        return []
    approx_of = dict(zip(st["candidates"].tolist(), st["approx"].tolist()))
    return [(approx_of[d], float(e), d + base) for d, e in zip(st["rerank"].tolist(), st["exact"].tolist())]
