"""Index mutation: append documents / delete documents (host-side, off the hot path).

The reference's update policy (python/fast_plaid/search/update.py:65-452, rust/index/update.rs:30-473,
rust/index/delete.rs:26-145): create-if-missing; rebuild-from-scratch while the index is small and the
raw ``embeddings.npy`` is still around; otherwise the outlier buffer.  Documents are appended with the
existing codec and their raw embeddings kept in ``buffer.npy`` until ``buffer_size`` of them have
accumulated; then the buffered documents are deleted, the tokens of buffer + new documents that lie
farther than ``cluster_threshold`` from every centroid are clustered into new centroids appended to the
codebook (``update_centroids``), all of them are re-added with the expanded codec and the threshold is
re-estimated from their residuals.  Deletion rewrites the chunk files, renumbers the documents and
rebuilds the IVF.

The outlier search, min_k |x - c_k|^2 > threshold^2 over every token, runs on the tcgen05 nearest-centroid
kernel (``engine.nearest_centroid``) on a CUDA device with dim 128, and as the reference's dense torch
formula (update.py:144-150) elsewhere.
"""

from __future__ import annotations

import json
import math
import os
from typing import Any

import numpy as np
import torch

from . import build, store


def _load_raw(path: str) -> list[torch.Tensor]:
    arr = np.load(path, allow_pickle=True)
    return [torch.from_numpy(a) for a in arr]


def process_update(fp: Any, docs: list[torch.Tensor], metadata: list[dict] | None, batch_size: int,
                   kmeans_niters: int, max_points_per_centroid: int, n_samples_kmeans: int | None, seed: int,
                   start_from_scratch: int, buffer_size: int) -> None:
    index_path = fp.index
    meta = store.read_metadata(index_path)
    if meta is None:  # update.py:271-290
        fp.create(docs, kmeans_niters=kmeans_niters, max_points_per_centroid=max_points_per_centroid,
                  n_samples_kmeans=n_samples_kmeans, batch_size=batch_size, seed=seed, metadata=metadata)
        return
    n_old = int(meta.get("num_documents", 0))
    emb_path = os.path.join(index_path, "embeddings.npy")
    db = os.path.join(index_path, "metadata.db")
    if os.path.exists(db):
        # update.py:300-311: once a metadata table exists EVERY added document gets a row (an empty one when
        # no metadata is given), so that `_subset_` stays equal to the document id
        if metadata is None:
            metadata = [{} for _ in docs]
        if len(metadata) != len(docs):
            raise ValueError(
                f"The length of metadata ({len(metadata)}) must match the number of "
                f"documents_embeddings ({len(docs)})."
            )
        from ..filtering import update as _meta_update

        _meta_update(index=index_path, metadata=metadata)
    if n_old <= start_from_scratch and os.path.exists(emb_path):  # update.py:314-349
        old = _load_raw(emb_path)
        keep_db = os.path.exists(db)
        if keep_db:  # create() clears the directory's table: park it
            os.replace(db, db + ".keep")
        try:
            fp.create(old + docs, kmeans_niters=kmeans_niters, max_points_per_centroid=max_points_per_centroid,
                      nbits=int(meta["nbits"]), n_samples_kmeans=n_samples_kmeans, batch_size=batch_size, seed=seed,
                      start_from_scratch=start_from_scratch + 1,
                      compress_only=bool(meta.get("compress_only", False)))
        finally:
            if keep_db and os.path.exists(db + ".keep"):
                os.replace(db + ".keep", db)
        if len(old) + len(docs) > start_from_scratch and os.path.exists(emb_path):
            os.remove(emb_path)
        return
    from ..search.fast_plaid import save_list_tensors_on_disk

    device = fp.devices[0]
    buffer_path = os.path.join(index_path, "buffer.npy")
    buffered = _load_raw(buffer_path) if os.path.exists(buffer_path) else []
    if len(buffered) + len(docs) < buffer_size:  # update.py:431-445
        save_list_tensors_on_disk(buffer_path, buffered + docs)
        append_documents(index_path, docs, batch_size=batch_size, device=device)
        return
    # update.py:380-429: the buffered documents leave the index (their metadata rows stay: they come back with the
    # same ids) and are re-added together with the new ones once the codebook has grown
    if buffered:
        fp._delete_documents(list(range(n_old - len(buffered), n_old)), delete_metadata=False, delete_buffer=False)
        docs = buffered + docs
    threshold = float(np.load(os.path.join(index_path, "cluster_threshold.npy")).item())
    update_centroids(index_path, docs, threshold, device, kmeans_niters, max_points_per_centroid, seed,
                     n_samples_kmeans)
    if os.path.exists(buffer_path):
        os.remove(buffer_path)
    append_documents(index_path, docs, batch_size=batch_size, device=device, update_threshold=True)


@torch.inference_mode()
def outlier_mask(flat: torch.Tensor, centroids: torch.Tensor, cluster_threshold: float, device: str,
                 rows: int = 4096) -> torch.Tensor:
    """Host bool [n]: min_k |x - c_k|^2 > cluster_threshold^2 (update.py:121-150).

    On CUDA with dim 128 the distances come from the tcgen05 kernel (fp16 tokens and centroids, fp32 accumulation).
    Elsewhere they are the reference's x2 + y2 - 2 x.c in the tokens' dtype, in `rows`-row batches."""
    dev = torch.device(device)
    threshold_sq = cluster_threshold**2
    if dev.type == "cuda" and flat.shape[1] == 128:
        from ..engine import nearest_centroid

        _, dist2 = nearest_centroid(flat, centroids.to(dev))
        return (dist2 > threshold_sq).cpu()
    cent = centroids.to(device=dev, dtype=flat.dtype)
    y2 = torch.sum(cent**2, dim=1)
    mask = torch.zeros(flat.shape[0], dtype=torch.bool)
    for i in range(0, flat.shape[0], rows):
        batch = flat[i : i + rows].to(dev)
        x2 = torch.sum(batch**2, dim=1, keepdim=True)
        dists_sq = x2 + y2 - 2 * torch.matmul(batch, cent.T)
        mask[i : i + rows] = (torch.min(dists_sq, dim=1).values > threshold_sq).cpu()
    return mask


@torch.inference_mode()
def update_centroids(index_path: str, docs: list[torch.Tensor], cluster_threshold: float, device: str,
                     kmeans_niters: int, max_points_per_centroid: int, seed: int,
                     n_samples_kmeans: int | None) -> None:
    """Grow the codebook with k-means centroids of the outlier tokens (update.py:65-203).  Appends
    ``k_update = max(1, 4 * ceil(n_outliers / max_points_per_centroid))`` centroids to ``centroids.npy`` (float32, as
    the reference writes it), zero-length lists to ``ivf_lengths.npy`` and sets ``num_partitions``; without outliers
    the directory is left untouched."""
    centroids_path = os.path.join(index_path, "centroids.npy")
    if not os.path.exists(centroids_path):
        return
    existing = np.load(centroids_path)
    # the buffered documents come from disk, the new ones may be CUDA tensors
    flat = torch.cat([d.reshape(-1, existing.shape[1]).to(device) for d in docs])
    mask = outlier_mask(flat, torch.from_numpy(existing), cluster_threshold, device)
    outliers = flat[mask.to(flat.device)]
    n_out = int(outliers.shape[0])
    if n_out == 0:
        return
    k_update = max(1, math.ceil(n_out / max_points_per_centroid) * 4)
    new = build.compute_kmeans(outliers, int(outliers.shape[1]), device, kmeans_niters, max_points_per_centroid, seed,
                               n_samples_kmeans, num_partitions=k_update)
    new_np = new.detach().cpu().numpy().astype(np.float32)
    final = np.concatenate([existing, new_np], axis=0)
    np.save(centroids_path, final)
    ivf_path = os.path.join(index_path, "ivf_lengths.npy")
    if os.path.exists(ivf_path):
        lengths = np.load(ivf_path)
        np.save(ivf_path, np.concatenate([lengths, np.zeros(new_np.shape[0], dtype=lengths.dtype)]))
    meta_path = os.path.join(index_path, "metadata.json")
    with open(meta_path) as f:
        meta = json.load(f)
    meta["num_partitions"] = int(final.shape[0])
    with open(meta_path, "w") as f:
        json.dump(meta, f, indent=4)


def updated_threshold(index_path: str, old_num_embeddings: int, residual_norms: torch.Tensor) -> None:
    """update.rs:277-297: the 0.75 quantile of the appended tokens' residual norms, averaged with the stored threshold
    weighted by token counts (the stored one counts the `old_num_embeddings` tokens the index held before the append);
    written to ``cluster_threshold.npy`` as a float64 scalar."""
    new_count = int(residual_norms.shape[0])
    new_val = float(build._quantile_kth(residual_norms, 0.75))
    path = os.path.join(index_path, "cluster_threshold.npy")
    if os.path.exists(path):
        old_val = float(np.load(path).item())
        val = (old_val * old_num_embeddings + new_val * new_count) / (old_num_embeddings + new_count)
    else:
        val = new_val
    np.save(path, np.array(val, dtype=np.float64))


@torch.inference_mode()
def append_documents(index_path: str, docs: list[torch.Tensor], batch_size: int, device: str,
                     update_threshold: bool = False) -> None:
    """Encode with the codec on disk and append as new chunk(s) (update.rs:30-473); with `update_threshold` the
    cluster threshold is re-estimated from the appended tokens' residuals (update.rs:277-297)."""
    meta = store.read_metadata(index_path)
    nbits = int(meta["nbits"])
    dev = torch.device(device)
    cent = torch.from_numpy(np.load(os.path.join(index_path, "centroids.npy"))).to(dev, torch.float16)
    cutoffs = torch.from_numpy(np.load(os.path.join(index_path, "bucket_cutoffs.npy"))).to(dev)
    dim = int(cent.shape[1])
    cent_t = cent.t().contiguous()
    n_chunks = int(meta["num_chunks"])
    emb_offset = int(meta["num_embeddings"])
    n_docs = int(meta["num_documents"])
    per_chunk = max(1, int(batch_size))
    norms: list[torch.Tensor] = []
    for s in range(0, len(docs), per_chunk):
        chunk_docs = docs[s : s + per_chunk]
        lens = [int(d.shape[0]) for d in chunk_docs]
        flat = torch.cat([d.reshape(-1, dim).to(dev, torch.float16) for d in chunk_docs])
        codes_parts, res_parts = [], []
        for r in range(0, flat.shape[0], max(1, batch_size)):
            x = flat[r : r + batch_size]
            c, rr = build.encode(x, cent, cent_t, cutoffs, nbits)
            if update_threshold:  # fp32 norms of the fp16 residuals (update.rs:141-146)
                norms.append((x - cent.index_select(0, c)).float().norm(dim=1).cpu())
            codes_parts.append(c.cpu())
            res_parts.append(rr.cpu())
        codes = torch.cat(codes_parts) if codes_parts else torch.empty(0, dtype=torch.int64)
        res = torch.cat(res_parts) if res_parts else torch.empty((0, dim * nbits // 8), dtype=torch.uint8)
        store.write_chunk(index_path, n_chunks, codes, res, lens, emb_offset)
        n_chunks += 1
        emb_offset += int(codes.shape[0])
        n_docs += len(lens)
    if norms:
        updated_threshold(index_path, int(meta["num_embeddings"]), torch.cat(norms))
    compress_only = bool(meta.get("compress_only", False))
    if not compress_only:
        _rebuild_ivf(index_path, n_chunks, int(meta.get("num_partitions", cent.shape[0])), dev)
    store.write_metadata(index_path, num_chunks=n_chunks, nbits=nbits,
                         num_partitions=int(meta.get("num_partitions", cent.shape[0])),
                         num_embeddings=emb_offset, num_documents=n_docs, compress_only=compress_only)


def _rebuild_ivf(index_path: str, n_chunks: int, n_cells: int, dev: torch.device) -> None:
    codes, lens = [], []
    for i in range(n_chunks):
        cp = os.path.join(index_path, f"{i}.codes.npy")
        if os.path.exists(cp):
            codes.append(torch.from_numpy(np.load(cp)))
    lens = store.read_doclens(index_path, n_chunks)
    all_codes = torch.cat(codes) if codes else torch.empty(0, dtype=torch.int64)
    ivf, ivf_lengths = build.build_ivf(all_codes.to(dev), torch.tensor(lens, dtype=torch.int64), n_cells)
    store.write_ivf(index_path, ivf, ivf_lengths)


@torch.inference_mode()
def delete_from_index(index_path: str, subset: list[int], device: str) -> None:
    """delete.rs:26-145: drop the documents, keep the chunk structure, rebuild the IVF."""
    meta = store.read_metadata(index_path)
    if meta is None:
        raise RuntimeError("Failed to delete from index: metadata.json not found")
    n_chunks = int(meta["num_chunks"])
    drop = set(int(i) for i in subset)
    doc_base = 0
    emb_offset = 0
    n_docs = 0
    for i in range(n_chunks):
        dl_path = os.path.join(index_path, f"doclens.{i}.json")
        if not os.path.exists(dl_path):
            continue
        with open(dl_path) as f:
            lens = json.load(f)
        codes = torch.from_numpy(np.load(os.path.join(index_path, f"{i}.codes.npy")))
        res = torch.from_numpy(np.load(os.path.join(index_path, f"{i}.residuals.npy")))
        keep_doc = torch.tensor([(doc_base + j) not in drop for j in range(len(lens))], dtype=torch.bool)
        lens_t = torch.tensor(lens, dtype=torch.int64)
        keep_tok = torch.repeat_interleave(keep_doc, lens_t)
        new_lens = lens_t[keep_doc].tolist()
        store.write_chunk(index_path, i, codes[keep_tok], res[keep_tok], new_lens, emb_offset)
        emb_offset += int(keep_tok.sum())
        n_docs += len(new_lens)
        doc_base += len(lens)
    compress_only = bool(meta.get("compress_only", False))
    if not compress_only:
        _rebuild_ivf(index_path, n_chunks, int(meta.get("num_partitions", 1)), torch.device(device))
    store.write_metadata(index_path, num_chunks=n_chunks, nbits=int(meta["nbits"]),
                         num_partitions=int(meta.get("num_partitions", 1)), num_embeddings=emb_offset,
                         num_documents=n_docs, compress_only=compress_only)
