"""Every search-kernel variant against fp64 references with stated error bounds.

Which kernel runs depends on dim, nbits, the padded query width Qp = next_pow2(max(Q, 16)), the longest document of
the index and two process-wide pins (FPB_K1 / FPB_K5).  This file launches each variant:

  K1  v2 (tcgen05, dim 128, Qp <= 128), v1 (mma.sync) at D = 128 (Qp = 256, or pinned) and D = 64;
  K3  LPR = Qp / 8 from 2 to 32, one pass, two passes and every candidate scored, and the shuffle kernel that a
      code array without 16-byte alignment takes at LPR <= 4;
  K5  v4 (Qp 16 / 32), v5 (Qp 64 / 128, documents up to 16 384 tokens), the generic kernel for Qp = 256, for an index
      with one longer document and for every (dim, nbits) other than (128, 4).

The fp stages are checked entry by entry against intervals around fp64 values (tests/util.py, DESIGN.md "Parity
contract"): S, the per-token norms and every exact MaxSim score.  K5 is also run on its own, on re-rank lists written
by hand whose query tokens copy the boundary tokens of the listed documents (first, last, 8k+7, 8k+8, 159, 160), so a
dropped, repeated or misattributed token moves a score by far more than its interval.  The pinned fallback kernels
run in a child process (`python test_gpu_kernel_matrix.py --child OUT` with FPB_K1=v1 FPB_K5=v1), whose outputs the
parent checks with the same bounds.
"""

from __future__ import annotations

import ctypes
import os
import subprocess
import sys
import tempfile

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from util import (PAD_SENTINEL, build_oracle_index, centroid_score_bounds, dot_fp64, interval_report,  # noqa: E402
                  make_docs, make_queries, maxsim_bounds, normalise_like_the_kernels, to_index_tensors,
                  token_norm_bounds)

from oracle import plaid_oracle as po  # noqa: E402

pytestmark = pytest.mark.gpu

# document lengths at which the kernels change behaviour: the 8-token passes of v4 / v5, the 64-token tiles of the
# generic kernel, the 160-row tiles of v5, and v5's pass table (2048 passes = 16 384 tokens)
BOUNDARY_LENGTHS = [0, 1, 7, 8, 9, 15, 16, 17, 63, 64, 65, 159, 160, 161, 1023, 1024, 1025]
PLANTED_INDEXES = {
    # name: (dim, nbits, lengths added to BOUNDARY_LENGTHS)
    "short": (128, 4, []),
    "long": (128, 4, [16384]),  # v5 with one document per chunk
    "longer": (128, 4, [16384, 16385]),  # one document past v5's pass table: the whole index takes the generic kernel
    "short_d128_n2": (128, 2, []),
    "short_d64_n4": (64, 4, []),
    "short_d64_n2": (64, 2, []),  # the only decode with one lane per token
}
K_PLANTED = 2 * 128 + 5  # a partial last centroid tile of 5 rows
N_FULL = 52  # R = 13: not a multiple of v5's documents per chunk (4 here) nor of v4's document groups
NAN_BITS = 0x7FC0BEEF  # the pattern a slot keeps when K5 must not write it

Q_VALUES = [1, 15, 16, 17, 31, 32, 33, 64, 65, 100, 128, 129, 200, 256]
B_VALUES = [1, 3, 7]
PLANTED_CASES = (
    [("short", Q, B_VALUES[i % 3], i % 2 == 1) for i, Q in enumerate(Q_VALUES)]
    + [("long", Q, B_VALUES[i % 3], i % 2 == 0) for i, Q in enumerate([1, 17, 33, 65, 100, 128, 129, 256])]
    + [("longer", Q, B_VALUES[i % 3], i % 2 == 1) for i, Q in enumerate([17, 65, 128])]
    + [(name, Q, 3, i % 2 == 0) for name in ("short_d128_n2", "short_d64_n4", "short_d64_n2")
       for i, Q in enumerate([15, 100, 256])]
)
# the pinned fallbacks (child process): K1 v1 at D = 128 for Qp <= 128, the generic K5 where v4 / v5 would run
CHILD_CASES = [("short", 16, 3, False), ("short", 33, 7, True), ("short", 128, 3, False), ("long", 65, 3, True)]


def _case_id(c):
    return f"{c[0]}-Q{c[1]}-B{c[2]}" + ("-unnorm" if c[3] else "")


# ---- the planted index: explicit lengths, seeded random centroids and codes ------------------------------------
_planted: dict = {}


def _planted_index(name: str):
    """CPU tensors of the index plus its decoded (unnormalised) tokens; deterministic, so the child rebuilds it."""
    if name in _planted:
        return _planted[name]
    from fast_plaid_b200.engine import IndexTensors

    dim, nbits, extra = PLANTED_INDEXES[name]
    g = torch.Generator().manual_seed(1000 + dim + nbits + len(extra))
    lengths = BOUNDARY_LENGTHS + extra + torch.randint(1, 40, (24,), generator=g).tolist()
    T = sum(lengths)
    centroids = torch.nn.functional.normalize(torch.randn(K_PLANTED, dim, generator=g), dim=-1).half()
    # bucket weights like those of a trained index: sorted, roughly symmetric, a few hundredths
    bw = (torch.linspace(-1.6, 1.6, 2**nbits) * 0.035 + 0.002 * torch.randn(2**nbits, generator=g)).sort().values.half()
    codes = torch.randint(0, K_PLANTED, (T,), generator=g)
    residuals = torch.randint(0, 256, (T, dim * nbits // 8), generator=g, dtype=torch.uint8)
    lens = torch.tensor(lengths, dtype=torch.int64)
    N = len(lengths)
    ivf_lengths = torch.zeros(K_PLANTED, dtype=torch.int64)
    ivf_lengths[0] = N  # every document in cell 0: the K5-only runs never probe
    t = IndexTensors(nbits, centroids, bw, lens, codes, residuals, torch.arange(N), ivf_lengths)
    rev, lookup = po.codec_luts(nbits)
    e16 = po.decode_unnormalised(residuals, bw, rev, lookup, codes, centroids, dim, nbits)
    offs = [0]
    for n in lengths:
        offs.append(offs[-1] + n)
    _planted[name] = (t, e16, offs[:-1], lengths)
    return _planted[name]


def _planted_inputs(case):
    """Re-rank lists, their lengths and queries whose tokens copy boundary tokens of the listed documents."""
    name, Q, B, unnorm = case
    lengths = _planted_index(name)[3]
    R = N_FULL // 4
    N = len(lengths)
    g = torch.Generator().manual_seed(7 * Q + B + (100 if unnorm else 0))
    longest = max(range(N), key=lambda d: lengths[d])
    pool = [d for d in range(N) if d != longest]
    lists, n_rer = [], []
    for b in range(B):
        lst = [longest] + [pool[(5 * b + Q + i) % len(pool)] for i in range(R - 1)]
        lst[3] = lst[1]  # a repeated document
        lst[4] = 0  # the empty document
        if name == "longer":
            lst[2] = longest - 1  # both long documents
        lists.append(lst)
        n_rer.append(0 if b == 2 else (R if b % 2 == 0 else R - 1 - b % 4))
    return lists, n_rer, g


def _planted_queries(case, norms16: torch.Tensor) -> torch.Tensor:
    name, Q, B, unnorm = case
    t, e16, offs, lengths = _planted_index(name)
    lists, n_rer, g = _planted_inputs(case)
    ehat = normalise_like_the_kernels(e16, norms16)
    dim = e16.shape[1]
    out = torch.empty(B, Q, dim)
    for b in range(B):
        docs = [d for d in (lists[b][: n_rer[b]] or lists[b]) if lengths[d] > 0]
        for j in range(Q):
            d = docs[j % len(docs)]
            n = lengths[d]
            pos = [p for p in (0, n - 1, 7, 8, 8 * (n // 16) + 7, 8 * (n // 16) + 8, 159, 160) if p < n]
            row = offs[d] + pos[(j // len(docs)) % len(pos)]
            v = torch.nn.functional.normalize(ehat[row].float() + 0.05 * torch.randn(dim, generator=g), dim=0)
            out[b, j] = v * (11.0 if unnorm else 1.0)
    return out.half()


def _gpu_planted(case, device: str) -> dict:
    """K1 on the queries, then K5 alone on the hand-written re-rank lists; everything the checks need, on the CPU."""
    from fast_plaid_b200.engine import DeviceIndex

    didx = _planted_device(case[0], device)
    norms = didx.token_norms[: didx.num_tokens].cpu()
    q16 = _planted_queries(case, norms)
    lists, n_rer, _ = _planted_inputs(case)
    params = DeviceIndex.make_params(10, N_FULL, 8)
    q = q16.to(device)
    st = didx.run_stages(q, params, upto="centroid_scores")
    R = st["layout"].R
    st["rerank"].copy_(torch.tensor(lists, dtype=torch.int32))
    st["n_rerank"].copy_(torch.tensor(n_rer, dtype=torch.int32))
    st["exact"].view(torch.int32).fill_(NAN_BITS)
    didx.stage_fn("maxsim", q, params)()
    torch.cuda.synchronize()
    assert R == len(lists[0])
    return {"S": st["S"].cpu(), "tmax": st["tmax"].cpu(), "exact": st["exact"].cpu(), "norms": norms, "q16": q16}


_planted_dev: dict = {}


def _planted_device(name: str, device: str):
    from fast_plaid_b200.engine import DeviceIndex

    if name not in _planted_dev:
        _planted_dev.clear()  # one planted index resident at a time
        _planted_dev[name] = DeviceIndex(_planted_index(name)[0], device)
    return _planted_dev[name]


# ---- checks shared by the planted cases, the pipeline cases and the child's outputs ----------------------------
def _check_centroid_scores(S: torch.Tensor, tmax: torch.Tensor, centroids16: torch.Tensor, q16: torch.Tensor) -> None:
    """S [B, K, Qp] within the fp64 interval, padded columns exactly 0; tmax the max of S over each 128-row tile."""
    B, Q = q16.shape[0], q16.shape[1]
    K = centroids16.shape[0]
    for b in range(B):
        lo, hi, x, g = centroid_score_bounds(centroids16, q16[b])
        msg = interval_report(S[b, :, :Q], lo, hi, x, g)
        assert not msg, f"query {b}: S: {msg}"
    assert bool((S[:, :, Q:] == 0).all()), "a padded query column of S is not 0"
    n_tiles = tmax.shape[2]
    Sf = torch.full((B, n_tiles * 128, S.shape[2]), float("-inf"))
    Sf[:, :K] = S.float()
    ref = Sf.view(B, n_tiles, 128, S.shape[2]).amax(2).transpose(1, 2).half()
    assert torch.equal(ref, tmax), "tmax is not the maximum of S over the valid rows of each centroid tile"


def _check_norms(norms16: torch.Tensor, e16: torch.Tensor) -> None:
    lo, hi = token_norm_bounds(e16)
    bad = (norms16 < lo) | (norms16 > hi)
    assert not bool(bad.any()), f"{int(bad.sum())} token norms outside their fp64 interval (first at {int(bad.nonzero()[0])})"


def _check_exact(got: torch.Tensor, ehat_dev: torch.Tensor, offs: list[int], lengths: list[int],
                 q16: torch.Tensor, lists: list[list[int]], n_rer: list[int], what: str, nan_tail: bool = True) -> None:
    """exact[b, r] for r < n_rer[b] inside the fp64 interval of document lists[b][r]; with `nan_tail`, the slots past
    n_rer[b] still hold NAN_BITS."""
    for b in range(len(lists)):
        n = n_rer[b]
        x, g = dot_fp64(ehat_dev, q16[b].to(ehat_dev.device))
        bounds = maxsim_bounds(ehat_dev, [offs[d] for d in lists[b][:n]], [lengths[d] for d in lists[b][:n]],
                               q16[b].to(ehat_dev.device), x, g)
        for r, (lo, hi) in enumerate(bounds):
            s = float(got[b, r])
            d = lists[b][r]
            if lengths[d] == 0:
                assert s == q16.shape[1] * PAD_SENTINEL, f"{what}: query {b} slot {r}: empty document scored {s}"
            assert lo <= s <= hi, f"{what}: query {b} slot {r} (doc {d}, {lengths[d]} tokens): {s} outside [{lo}, {hi}]"
        if nan_tail and n < got.shape[1]:
            tail = got[b, n:].view(torch.int32)
            assert bool((tail == NAN_BITS).all()), f"{what}: query {b}: a slot at or past n_rerank = {n} was written"


def _check_planted(case, out: dict, device: str) -> None:
    name = case[0]
    t, e16, offs, lengths = _planted_index(name)
    lists, n_rer, _ = _planted_inputs(case)
    _check_centroid_scores(out["S"], out["tmax"], t.centroids, out["q16"])
    _check_norms(out["norms"], e16)
    ehat = normalise_like_the_kernels(e16, out["norms"]).to(device)
    _check_exact(out["exact"], ehat, offs, lengths, out["q16"], lists, n_rer, _case_id(case))


@pytest.mark.parametrize("case", PLANTED_CASES, ids=_case_id)
def test_maxsim_with_planted_maxima(case, cuda_device):
    _check_planted(case, _gpu_planted(case, cuda_device), cuda_device)


# ---- the pinned fallback kernels, in a child process ---------------------------------------------------------
def _child(out_path: str) -> None:
    torch.save({_case_id(c): _gpu_planted(c, "cuda:0") for c in CHILD_CASES}, out_path)


def test_pinned_fallback_kernels_in_a_child_process(cuda_device):
    """FPB_K1=v1 FPB_K5=v1 are read once per process: K1 v1 at D = 128 for Qp <= 128 and the generic K5 where v4 /
    v5 would run are reached in a child, whose outputs get the same checks."""
    with tempfile.TemporaryDirectory() as tmp:
        out_path = os.path.join(tmp, "child.pt")
        env = dict(os.environ, FPB_K1="v1", FPB_K5="v1")
        proc = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", out_path], env=env,
                              capture_output=True, text=True, timeout=600)
        assert proc.returncode == 0, f"child failed:\n{proc.stdout[-3000:]}\n{proc.stderr[-3000:]}"
        outs = torch.load(out_path)
    for c in CHILD_CASES:
        _check_planted(c, outs[_case_id(c)], cuda_device)


# ---- the whole pipeline over the shapes the other parity tests do not reach ----------------------------------
PIPE_DIMS = [(128, 4), (128, 2), (64, 4), (64, 2)]
PIPE_CASES = [(dim, nbits, Q, 8) for dim, nbits in PIPE_DIMS for Q in (17, 33, 129, 256)] + [
    (128, 4, 33, 1), (128, 4, 129, 32)]

_pipe: dict = {}


def _pipeline_index(dim: int, nbits: int, device: str):
    key = (dim, nbits)
    if key not in _pipe:
        from fast_plaid_b200.engine import DeviceIndex

        docs = make_docs(300, 5, 120, dim=dim, seed=77 + dim + nbits)
        oidx, _ = build_oracle_index(docs, nbits=nbits, kmeans_niters=3)
        didx = DeviceIndex(to_index_tensors(oidx), device)
        T = int(oidx.doc_offsets[-1])
        e16 = po.decode_unnormalised(oidx.doc_residuals[:T], oidx.bucket_weights, oidx.byte_reversed_bits_map,
                                     oidx.bucket_weight_indices_lookup, oidx.doc_codes[:T], oidx.centroids, dim, nbits)
        _pipe[key] = (oidx, didx, docs, e16)
    return _pipe[key]


def _snapshot(st: dict) -> dict:
    return {k: (v.clone() if isinstance(v, torch.Tensor) else v) for k, v in st.items() if k != "workspace"}


@pytest.mark.parametrize("case", PIPE_CASES, ids=lambda c: f"d{c[0]}-n{c[1]}-Q{c[2]}-probe{c[3]}")
def test_pipeline_over_all_kernel_shapes(case, cuda_device):
    from fast_plaid_b200.engine import (FPB_FLAG_APPROX_DIRECT, FPB_FLAG_APPROX_EXACT_ALL, FPB_FLAG_APPROX_TWO_PASS,
                                        DeviceIndex)

    dim, nbits, Q, n_probe = case
    oidx, didx, docs, e16 = _pipeline_index(dim, nbits, cuda_device)
    B = 3
    queries = make_queries(B, Q, dim=dim, seed=Q + n_probe, docs=docs)
    q16 = queries.half()
    params = DeviceIndex.make_params(10, 64, n_probe)
    runs = {}
    for flag in (FPB_FLAG_APPROX_EXACT_ALL, FPB_FLAG_APPROX_DIRECT, FPB_FLAG_APPROX_TWO_PASS):
        runs[flag] = _snapshot(didx.run_stages(q16.to(cuda_device), DeviceIndex.with_flags(params, flag)))
    torch.cuda.synchronize()
    st = {k: (v.cpu() if isinstance(v, torch.Tensor) else v) for k, v in runs[FPB_FLAG_APPROX_EXACT_ALL].items()}

    # integer stages bit-exact against the canonical oracle fed the GPU's S
    for b in range(B):
        S_b = st["S"][b, :, :Q].contiguous()
        ref = po.search_one(queries[b], oidx, n_probe, 2000, params.n_full_scores, params.top_k, ties="canonical",
                            return_stages=True, inject={"S": S_b})
        cells = torch.unique(st["cells"][b].flatten().long())
        assert torch.equal(cells[cells >= 0], ref["cells"]), f"query {b}: probed cells differ"
        n = int(st["n_cand"][b])
        assert torch.equal(st["cand"][b, :n].long(), ref["candidates"]), f"query {b}: candidate ids differ"
        approx = st["approx"][b, :n]
        if not torch.equal(approx, ref["approx"]):
            # an fp32 partial sum past 24 bits rounds differently in ATen's vectorised order: prune on the GPU's
            rel = ((approx - ref["approx"]).abs() / ref["approx"].abs().clamp_min(1.0)).max()
            assert float(rel) < 1e-6, f"query {b}: approximate scores differ by {float(rel)}"
            ref = po.search_one(queries[b], oidx, n_probe, 2000, params.n_full_scores, params.top_k,
                                ties="canonical", return_stages=True, inject={"S": S_b, "approx": approx})
        r = int(st["n_rerank"][b])
        assert torch.equal(st["rerank"][b, :r].long(), ref["rerank"]), f"query {b}: pruned list differs"

    # the three approximate-stage modes give the same pruned lists, re-rank scores and results
    for flag in (FPB_FLAG_APPROX_DIRECT, FPB_FLAG_APPROX_TWO_PASS):
        other = runs[flag]
        for b in range(B):
            r = int(st["n_rerank"][b])
            assert int(other["n_rerank"][b]) == r
            assert torch.equal(other["rerank"][b, :r].cpu(), st["rerank"][b, :r]), f"flag {flag} query {b}: pruned list"
            assert torch.equal(other["rerank_approx"][b, :r].cpu(), st["rerank_approx"][b, :r])
            assert torch.equal(other["exact"][b, :r].cpu(), st["exact"][b, :r])
        for k in ("ids", "scores", "counts"):
            assert torch.equal(other[k].cpu(), st[k]), f"flag {flag}: {k} differ"

    # fp stages inside their fp64 intervals
    _check_centroid_scores(st["S"], st["tmax"], oidx.centroids, q16)
    norms = didx.token_norms[: didx.num_tokens].cpu()
    _check_norms(norms, e16)
    ehat = normalise_like_the_kernels(e16, norms).to(cuda_device)
    offs = oidx.doc_offsets.tolist()
    lengths = oidx.doc_lengths.tolist()
    n_rer = [int(x) for x in st["n_rerank"]]
    lists = [st["rerank"][b, : n_rer[b]].tolist() for b in range(B)]
    _check_exact(st["exact"][:, : max(n_rer)], ehat, offs, lengths, q16, lists, n_rer, f"pipeline {case}",
                 nan_tail=False)


# ---- a code array without 16-byte alignment -------------------------------------------------------------------
@pytest.mark.parametrize("Q", [9, 17])
def test_misaligned_doc_codes_give_the_same_bytes(Q, cuda_device):
    """The shuffle-free K3 kernel loads codes as int2 / int4 and is only launched on a 16-byte-aligned code array; an
    index whose doc_codes is the view [1:] of a longer int32 tensor takes the shuffle kernel (LPR 2 and 4), and every
    stage must give the same bytes as on the aligned index."""
    from fast_plaid_b200.engine import FPB_FLAG_APPROX_DIRECT, FPB_FLAG_APPROX_TWO_PASS, DeviceIndex, _check, _ptr

    oidx, didx, docs, _ = _pipeline_index(128, 4, cuda_device)
    mis = DeviceIndex(to_index_tensors(oidx), cuda_device)
    base = torch.zeros(mis.doc_codes.numel() + 1, dtype=torch.int32, device=mis.device)
    base[1:].copy_(mis.doc_codes)
    codes = base[1:]
    assert codes.data_ptr() % 16 != 0
    torch.cuda.synchronize()
    mis._lib.fpb_index_destroy(mis._handle)
    handle = ctypes.c_void_p()
    _check(mis._lib.fpb_index_create(
        ctypes.byref(handle), mis.device.index, mis.nbits, mis.dim, mis.num_centroids, _ptr(mis.centroids),
        _ptr(mis.bucket_weights), mis.num_documents, _ptr(mis.doc_offsets), _ptr(codes), _ptr(mis.doc_residuals),
        _ptr(mis.token_norms), _ptr(mis.ivf_offsets), _ptr(mis.ivf_pids), int(mis.ivf_pids.numel()), mis.max_doc_len,
        0))
    mis._handle = handle
    mis.doc_codes = codes
    mis._codes_base = base  # keeps the storage alive
    queries = make_queries(3, Q, seed=Q, docs=docs).half().to(cuda_device)
    for flag in (FPB_FLAG_APPROX_DIRECT, FPB_FLAG_APPROX_TWO_PASS):
        params = DeviceIndex.with_flags(DeviceIndex.make_params(10, 64, 8), flag)
        a = _snapshot(didx.run_stages(queries, params))
        m = _snapshot(mis.run_stages(queries, params))
        torch.cuda.synchronize()
        for k in ("S", "cells", "n_cand", "cand", "approx", "n_rerank", "rerank", "rerank_approx", "exact", "ids",
                  "scores", "counts"):
            x, y = a[k], m[k]
            if k in ("cand", "approx"):
                x = torch.cat([x[b, : int(a["n_cand"][b])] for b in range(3)])
                y = torch.cat([y[b, : int(m["n_cand"][b])] for b in range(3)])
            elif k in ("rerank", "rerank_approx", "exact"):
                x = torch.cat([x[b, : int(a["n_rerank"][b])] for b in range(3)])
                y = torch.cat([y[b, : int(m["n_rerank"][b])] for b in range(3)])
            assert torch.equal(x, y), f"flag {flag}: {k} differs on the misaligned code array"
    mis.close()


if __name__ == "__main__":
    if len(sys.argv) == 3 and sys.argv[1] == "--child":
        _child(sys.argv[2])
