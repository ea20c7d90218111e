"""CPU oracle for index updates (the centroid expansion of the update path).
TEST INFRASTRUCTURE ONLY -- see the header of ``plaid_oracle.py`` for the import rules.

Restates, op for op in PyTorch-CPU, ``update_centroids`` (python/fast_plaid/search/update.py:65-203) on in-memory
arrays and the cluster-threshold update of ``update_index`` (rust/index/update.rs:141-146, :277-297).
"""

from __future__ import annotations

import math

import numpy as np
import torch

from .index_oracle import scalar_quantile_kthvalue


def update_centroids(centroids: np.ndarray, ivf_lengths: np.ndarray | None, meta: dict, new_embeddings,
                     cluster_threshold: float, max_points_per_centroid: int, kmeans_fn, rows: int = 4096) -> dict:
    """update_centroids (python/fast_plaid/search/update.py:65-203) on in-memory arrays, torch distance branch
    (:143-150): a token is an outlier when min_k |x - c_k|^2 > threshold^2, computed as x2 + y2 - 2 x.c in the
    tokens' dtype in `rows`-row batches; k_update = max(1, 4 * ceil(n_outliers / max_points_per_centroid)) new
    centroids from `kmeans_fn(outliers, k_update)` are appended (float32), the IVF gets zero-length lists and
    num_partitions the new K.  Returns the outlier mask, k_update (None without outliers) and the new arrays."""
    flat = torch.cat(list(new_embeddings)) if isinstance(new_embeddings, (list, tuple)) else new_embeddings
    cent = torch.from_numpy(centroids).to(flat.dtype)
    y2 = torch.sum(cent**2, dim=1)
    mask = torch.zeros(flat.shape[0], dtype=torch.bool)
    for i in range(0, flat.shape[0], rows):
        b = flat[i : i + rows]
        d = torch.sum(b**2, dim=1, keepdim=True) + y2 - 2 * torch.matmul(b, cent.T)
        mask[i : i + rows] = torch.min(d, dim=1).values > cluster_threshold**2
    out = {"mask": mask, "k_update": None, "centroids": centroids, "ivf_lengths": ivf_lengths,
           "num_partitions": meta.get("num_partitions")}
    n_out = int(mask.sum())
    if n_out == 0:
        return out
    k_update = max(1, math.ceil(n_out / max_points_per_centroid) * 4)
    new = kmeans_fn(flat[mask], k_update).detach().cpu().numpy().astype(np.float32)
    out["k_update"] = k_update
    out["centroids"] = np.concatenate([centroids, new], axis=0)
    if ivf_lengths is not None:
        out["ivf_lengths"] = np.concatenate([ivf_lengths, np.zeros(new.shape[0], dtype=ivf_lengths.dtype)])
    out["num_partitions"] = int(out["centroids"].shape[0])
    return out


def updated_threshold(old_threshold: float | None, old_num_embeddings: int, tokens: torch.Tensor,
                      centroids: torch.Tensor, codes: torch.Tensor) -> float:
    """The threshold update of update_index (rust/index/update.rs:141-146, :277-297): fp32 norms of the fp16
    residuals of the appended tokens, their 0.75 kthvalue quantile, averaged with the stored threshold weighted by
    the token counts (the stored one by num_embeddings as metadata.json held it before the append, :61)."""
    norms = (tokens.to(torch.float16) - centroids.to(torch.float16).index_select(0, codes)).float().norm(2, dim=1)
    new = float(scalar_quantile_kthvalue(norms, 0.75))
    if old_threshold is None:
        return new
    n = int(norms.shape[0])
    return (old_threshold * old_num_embeddings + new * n) / (old_num_embeddings + n)
