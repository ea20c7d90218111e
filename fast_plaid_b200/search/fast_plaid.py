"""The FastPlaid Python surface on top of the B200 engine.

Same class, method names, argument meaning and error behaviour as the reference's
``fast_plaid.search.FastPlaid`` (python/fast_plaid/search/fast_plaid.py:325-1186), same index
directory on disk, PyTorch tensors in and ``list[list[(doc_id, score)]]`` out.  What differs
is underneath: the whole query batch goes through one C-ABI call into hand-written sm_100a
kernels (``fast_plaid_b200/csrc``) instead of a per-query loop of ATen ops, and with several
GPUs the index is sharded by document (one process per GPU, NCCL all-gather of per-shard
records) instead of replicated.

There is no CPU search path: ``device="cpu"`` can build / update / delete an index directory
(host-side work) but ``search`` raises.
"""

from __future__ import annotations

import gc
import glob
import json
import math
import os
import threading
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path
from typing import Any

import numpy as np
import torch

try:  # same dependency as the reference (fast_plaid.py:20-21)
    from filelock import FileLock
    from filelock import Timeout as FileLockTimeout
except ImportError:  # pragma: no cover - filelock ships with the image
    FileLock = None  # type: ignore
    FileLockTimeout = Exception  # type: ignore

from .. import engine as _engine
from ..engine import DeviceIndex, IndexTensors
from ..index import build as _build
from ..index import store as _store


class _NullLock:
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False

    def acquire(self, timeout: float = -1):
        return self

    def release(self):
        pass


def save_list_tensors_on_disk(path: str, tensors: list[torch.Tensor]) -> None:
    """Pickled object array of raw document tensors (load.py:430-444)."""
    arr = np.empty(len(tensors), dtype=object)
    for i, t in enumerate(tensors):
        arr[i] = t.cpu().numpy()
    np.save(path, arr, allow_pickle=True)


try:  # CPython helper built next to the CUDA library (csrc/py/results.c); host glue only
    from .. import _fpb_results
except ImportError:  # pragma: no cover - the build produces it
    _fpb_results = None


def _results_to_lists(ids: torch.Tensor, scores: torch.Tensor, counts: torch.Tensor) -> list[list[tuple[int, float]]]:
    """Re-zip of search_on_device (fast_plaid.py:247-253): per query the first `count` (id, score) pairs.
    The 6 400 tuples of a 64 x 100 result are the dominant host cost of a search call: built in C when the
    helper is present (0.2 ms), else with one flat zip and B list slices (0.5 ms)."""
    k = int(ids.shape[1]) if ids.dim() == 2 else 0
    B = int(counts.shape[0])
    if (_fpb_results is not None and B > 0 and ids.device.type == "cpu" and ids.dtype == torch.int64
            and scores.dtype == torch.float32 and counts.dtype == torch.int32 and ids.is_contiguous()
            and scores.is_contiguous() and counts.is_contiguous()):
        return _fpb_results.zip_results(ids.data_ptr(), scores.data_ptr(), counts.data_ptr(), B, k)
    flat = list(zip(ids.reshape(-1).tolist(), scores.reshape(-1).tolist()))
    return [flat[b * k : b * k + n] for b, n in enumerate(counts.tolist())]


class FastPlaid:
    """Create, update and search a PLAID index; drop-in for the reference class."""

    def __init__(
        self,
        index: str,
        device: str | list[str] | None = None,
        low_memory: bool = True,
        shard: tuple[int, int] | str | None = None,
        query_groups: int = 1,
        **kwargs: Any,  # noqa: ARG002
    ) -> None:
        """``index``/``device``/``low_memory`` as in the reference (fast_plaid.py:328-385).

        ``low_memory`` is accepted and ignored: a B200 holds the whole index in HBM.
        ``shard``: ``(rank, world)`` makes this process one rank of the document-sharded search (one
        process per GPU; both exchanges are NCCL all-gathers issued below the C ABI, csrc/comm.cu);
        ``"auto"`` takes rank/world from an initialised process group.  ``query_groups`` (a divisor of
        world) arranges the ranks as query groups x document shards: each rank then holds
        1 / (world / query_groups) of the documents and searches 1 / query_groups of every batch.
        """
        self.devices = self._resolve_devices(device)

        self.index = index
        self.low_memory = low_memory
        if shard == "auto":
            import torch.distributed as dist

            shard = (dist.get_rank(), dist.get_world_size()) if dist.is_initialized() else None
        self.shard: tuple[int, int] | None = shard  # type: ignore[assignment]
        self.query_groups = int(query_groups)
        self._comm = None
        if self.shard is not None and len(self.devices) != 1:
            raise ValueError("sharded mode is one process per GPU: pass exactly one device")
        if self.shard is not None:
            _engine.shard_grid(self.shard[0], self.shard[1], self.query_groups)  # validates the grid

        if not os.path.exists(self.index):
            os.makedirs(self.index, exist_ok=True)
        self.lock_path = os.path.join(self.index, "plaid.lock")
        self.lock = FileLock(self.lock_path) if FileLock is not None else _NullLock()
        self._last_known_mtime = 0.0
        self._index_swap_lock = threading.Lock()
        self.indices: dict[str, DeviceIndex | None] = {}
        self._check_and_reload_index()

    # ------------------------------------------------------------------ lifetime
    def close(self) -> None:
        if getattr(self, "_comm", None) is not None:
            self._comm.close()
            self._comm = None
        with self._index_swap_lock:
            for idx in self.indices.values():
                if idx is not None:
                    idx.close()
            self.indices.clear()
        gc.collect()

    def __enter__(self) -> "FastPlaid":
        return self

    def __exit__(self, exc_type, exc_val, exc_tb) -> None:
        self.close()

    # ------------------------------------------------------------------ (re)loading
    def _update_mtime(self) -> None:
        meta_path = os.path.join(self.index, "metadata.json")
        if os.path.exists(meta_path):
            self._last_known_mtime = Path(meta_path).stat().st_mtime

    def _load_all(self) -> dict[str, DeviceIndex | None]:
        """disk -> CPU tensors -> one DeviceIndex per CUDA device (load.py:368-427)."""
        new: dict[str, DeviceIndex | None] = {d: None for d in self.devices}
        if not os.path.exists(os.path.join(self.index, "metadata.json")):
            return new
        if len(self.devices) == 1 and self.devices[0] != "cpu":
            # loader fast path: chunk files -> pinned staging -> HBM, only this shard's document range
            dev = self.devices[0]
            try:
                n_docs = read_num_documents(self.index)
                rng = None
                if self.shard is not None:
                    _, doc_shard, n_shards = _engine.shard_grid(self.shard[0], self.shard[1], self.query_groups)
                    rng = ((n_docs * doc_shard) // n_shards, (n_docs * (doc_shard + 1)) // n_shards)
                loaded = _store.read_index_to_device(self.index, dev, rng)
                if loaded is not None:
                    new[dev] = DeviceIndex(loaded[0], dev, doc_id_base=loaded[1])
            except Exception as e:  # load.py:393-399, :414-416
                print(f"Warning: Failed to load index on {dev}: {e}")
            self._host_data = None
            return new
        try:
            data = _store.read_index(self.index)
        except Exception as e:  # load.py:393-399
            print(f"Critical Error loading index from disk: {e}")
            return new
        if data is None:
            return new
        self._host_data = data if any(d == "cpu" for d in self.devices) else None
        base = 0
        if self.shard is not None:
            _, doc_shard, n_shards = _engine.shard_grid(self.shard[0], self.shard[1], self.query_groups)
            data, base = _engine.shard_tensors(data, doc_shard, n_shards)

        def provision(device: str):
            if device == "cpu":
                return device, None
            try:
                return device, DeviceIndex(data, device, doc_id_base=base)
            except Exception as e:  # load.py:414-416
                print(f"Warning: Failed to load index on {device}: {e}")
                return device, None

        if len(self.devices) == 1:
            dev, idx = provision(self.devices[0])
            new[dev] = idx
        else:
            with ThreadPoolExecutor(max_workers=len(self.devices)) as ex:
                new = dict(ex.map(provision, self.devices))
        return new

    def _check_and_reload_index(self, blocking: bool = True) -> bool:
        """Optimistic mtime check + double-checked reload under the file lock
        (fast_plaid.py:433-514)."""
        meta_path = os.path.join(self.index, "metadata.json")
        if not os.path.exists(meta_path):
            with self._index_swap_lock:
                for d in self.devices:
                    self.indices[d] = None
            return True
        current = Path(meta_path).stat().st_mtime
        if current <= self._last_known_mtime and self._loaded():
            return True
        if not blocking:
            try:
                self.lock.acquire(timeout=0)
            except FileLockTimeout:
                return False
            try:
                return self._reload_under_lock()
            finally:
                self.lock.release()
        with self.lock:
            return self._reload_under_lock()

    def _loaded(self) -> bool:
        return any(v is not None for v in self.indices.values()) or (
            self.devices == ["cpu"] and getattr(self, "_cpu_loaded", False)
        )

    def _reload_under_lock(self) -> bool:
        meta_path = os.path.join(self.index, "metadata.json")
        current = Path(meta_path).stat().st_mtime
        if current <= self._last_known_mtime and self._loaded():
            return True
        new = self._load_all()
        with self._index_swap_lock:
            old = self.indices
            self.indices = new
            self._last_known_mtime = current
            self._cpu_loaded = True
        self._retire(old)
        return True

    @staticmethod
    def _retire(old: dict) -> None:
        """A search thread may still hold a snapshot of the swapped-out handles (`_loaded_indices`): they are not
        closed here; DeviceIndex.__del__ frees the fpb_index and the HBM when the last reference goes away."""
        old.clear()
        gc.collect()

    def _swap_in_fresh(self) -> None:
        new = self._load_all()
        with self._index_swap_lock:
            old = self.indices
            self.indices = new
            self._update_mtime()
            self._cpu_loaded = True
        self._retire(old)

    # ------------------------------------------------------------------ create / update / delete
    @staticmethod
    def _resolve_devices(device: str | list[str] | None) -> list[str]:
        """Device list semantics of fast_plaid.py:350-362: one string, a list, or by default every
        visible GPU (else "cpu"); bare "cuda" means cuda:0; duplicates dropped, order kept.
        Anything that is not "cpu" / "cuda:N" is refused like parse_device (load.rs:16-37)."""
        if isinstance(device, str):
            wanted = [device]
        elif isinstance(device, list):
            wanted = list(device)
        else:
            n_gpu = torch.cuda.device_count() if torch.cuda.is_available() else 0
            wanted = [f"cuda:{i}" for i in range(n_gpu)] or ["cpu"]
        resolved: list[str] = []
        for d in wanted:
            d = "cuda:0" if d == "cuda" else d
            if d != "cpu" and not (d.startswith("cuda:") and d[5:].isdigit()):
                raise ValueError(f"Unsupported device string: '{d}'")
            if d not in resolved:
                resolved.append(d)
        return resolved

    def _format_embeddings(self, embeddings):
        if isinstance(embeddings, torch.Tensor):
            return embeddings.squeeze(0) if embeddings.dim() == 3 and embeddings.shape[0] == 1 else embeddings
        if not isinstance(embeddings, (list, tuple)) and hasattr(embeddings, "__getitem__") and hasattr(embeddings, "__len__"):
            return embeddings  # a lazy document sequence (e.g. index.synthetic.SyntheticDocuments): never materialised
        return [e.squeeze(0) if e.dim() == 3 else e for e in embeddings]

    @staticmethod
    def _prepare_index_directory(index_path: str) -> None:
        """fast_plaid.py:715-741"""
        if os.path.isdir(index_path):
            for pat in ("*.json", "*.npy"):
                for f in glob.glob(os.path.join(index_path, pat)):
                    try:
                        os.remove(f)
                    except OSError:
                        pass
        elif not os.path.exists(index_path):
            os.makedirs(index_path)

    @torch.inference_mode()
    def create(
        self,
        documents_embeddings: list[torch.Tensor] | torch.Tensor,
        kmeans_niters: int = 4,
        max_points_per_centroid: int = 256,
        nbits: int = 4,
        n_samples_kmeans: int | None = None,
        batch_size: int = 25_000,
        seed: int = 42,
        use_triton_kmeans: bool | None = None,  # noqa: ARG002  (no Triton in this build)
        metadata: list[dict[str, Any]] | None = None,
        start_from_scratch: int = 1000,
        compress_only: bool = False,
    ) -> "FastPlaid":
        """Create and save the index (fast_plaid.py:516-637)."""
        with self.lock:
            docs = self._format_embeddings(documents_embeddings)
            if isinstance(docs, torch.Tensor):
                docs = list(docs) if docs.dim() == 3 else [docs]
            num_docs = len(docs)
            self._prepare_index_directory(self.index)
            if metadata is not None:
                if len(metadata) != num_docs:
                    raise ValueError(
                        f"The length of metadata ({len(metadata)}) must match the number of "
                        f"documents_embeddings ({num_docs})."
                    )
                from ..filtering import create as _meta_create

                _meta_create(index=self.index, metadata=metadata)
            if num_docs <= start_from_scratch:
                save_list_tensors_on_disk(os.path.join(self.index, "embeddings.npy"), [docs[i] for i in range(num_docs)])
            dim = int(docs[0].shape[-1])
            _engine.check_supported(dim, nbits)  # fail before writing an index the engine cannot search
            primary = self.devices[0]
            centroids = _build.compute_kmeans(
                docs, dim, primary, kmeans_niters, max_points_per_centroid, seed, n_samples_kmeans
            )
            _build.create_index(docs, self.index, centroids, nbits=nbits, batch_size=batch_size, seed=seed,
                                compress_only=compress_only, device=primary)
            del centroids
            gc.collect()
            self._swap_in_fresh()
        return self

    @torch.inference_mode()
    def update(
        self,
        documents_embeddings: list[torch.Tensor] | torch.Tensor,
        metadata: list[dict[str, Any]] | None = None,
        batch_size: int = 25_000,
        kmeans_niters: int = 4,
        max_points_per_centroid: int = 256,
        n_samples_kmeans: int | None = None,
        seed: int = 42,
        start_from_scratch: int = 999,
        buffer_size: int = 100,
        use_triton_kmeans: bool | None = False,  # noqa: ARG002
    ) -> "FastPlaid":
        """Add documents (fast_plaid.py:640-713, update.py:206-452), with the reference's policy.

        Create-if-missing; while the index holds at most ``start_from_scratch`` documents it is
        rebuilt from the raw ``embeddings.npy`` plus the new documents.  Afterwards new documents
        are encoded with the existing codec and appended, and their raw embeddings are kept in
        ``buffer.npy``.  Once the buffer and the new documents reach ``buffer_size`` documents the
        buffered ones are deleted, the tokens farther than the cluster threshold from every
        centroid are clustered into new centroids appended to the codebook (update.py:65-203),
        all of them are re-added with the expanded codec, the threshold is re-estimated from
        their residuals and the buffer is removed.  ``use_triton_kmeans`` is accepted and ignored.
        """
        from ..index import update as _update

        with self.lock:
            docs = self._format_embeddings(documents_embeddings)
            if isinstance(docs, torch.Tensor):
                docs = list(docs) if docs.dim() == 3 else [docs]
            _update.process_update(self, docs, metadata, batch_size, kmeans_niters, max_points_per_centroid,
                                   n_samples_kmeans, seed, start_from_scratch, buffer_size)
            self._swap_in_fresh()
        return self

    @torch.inference_mode()
    def delete(self, subset: list[int], _delete_metadata: bool = True, _delete_buffer: bool = True) -> "FastPlaid":  # noqa: ARG002
        """Remove documents and renumber the rest (fast_plaid.py:1045-1157, delete.rs:26-145)."""
        with self.lock:
            self._delete_documents(subset, _delete_metadata, _delete_buffer)
            self._swap_in_fresh()
        return self

    def _delete_documents(self, subset: list[int], delete_metadata: bool, delete_buffer: bool) -> None:
        """The directory side of ``delete`` (the caller holds the lock and reloads the index afterwards)."""
        from ..index import update as _update

        # the buffer holds the raw embeddings of the most recent documents (fast_plaid.py:1084-1091): trim it like the
        # reference does (:1118-1145) so that a later update by either implementation does not resurrect deleted
        # documents
        buffer_path = os.path.join(self.index, "buffer.npy")
        if os.path.exists(buffer_path) and delete_buffer:
            n_docs = read_num_documents(self.index)
            buf = np.load(buffer_path, allow_pickle=True)
            start = n_docs - len(buf)
            drop_b = {i - start for i in subset if start <= i < n_docs}
            if drop_b:
                keep_b = [torch.from_numpy(buf[i]) for i in range(len(buf)) if i not in drop_b]
                if keep_b:
                    save_list_tensors_on_disk(buffer_path, keep_b)
                else:
                    os.remove(buffer_path)
        _update.delete_from_index(self.index, subset, device=self.devices[0])
        if os.path.exists(os.path.join(self.index, "metadata.db")) and delete_metadata:
            from ..filtering import delete as _meta_delete

            _meta_delete(index=self.index, subset=subset)
        emb_path = os.path.join(self.index, "embeddings.npy")
        if os.path.exists(emb_path):
            arr = np.load(emb_path, allow_pickle=True)
            drop = {i for i in subset if i < len(arr)}
            if drop:
                keep = [torch.from_numpy(arr[i]) for i in range(len(arr)) if i not in drop]
                if keep:
                    save_list_tensors_on_disk(emb_path, keep)
                else:
                    os.remove(emb_path)

    # ------------------------------------------------------------------ search
    def _loaded_indices(self) -> dict[str, Any]:
        """Snapshot of the per-device handles, reloading first if another process changed the
        directory (non-blocking try, then blocking if some device has no handle yet)."""
        for blocking in (False, True):
            self._check_and_reload_index(blocking=blocking)
            with self._index_swap_lock:
                snapshot = dict(self.indices)
            if all(h is not None for h in snapshot.values()):
                break
        return snapshot

    @staticmethod
    def _as_query_tensor(queries_embeddings) -> torch.Tensor:
        """A list of [Q_i, D] (or [1, Q_i, D]) tensors becomes one zero-padded [B, Qmax, D] tensor
        (fast_plaid.py:772-780).  A zero row scores 0 against every centroid, so -- exactly as in the reference --
        its "best" centroids are the first n_ivf_probe ones by the tie rule and it adds 0 to every document score."""
        if not isinstance(queries_embeddings, list):
            return queries_embeddings
        rows = [q.squeeze(0) if q.dim() == 3 else q for q in queries_embeddings]
        return torch.nn.utils.rnn.pad_sequence(rows, batch_first=True, padding_value=0.0)

    @staticmethod
    def _per_query_subsets(subset, num_queries: int):
        """`subset` may be None / [] (no filter), one id, one id list shared by all queries, or
        one list per query (fast_plaid.py:784-793)."""
        if subset is None or (isinstance(subset, list) and not subset):
            return None
        if isinstance(subset, int):
            subset = [subset]
        if isinstance(subset[0], int):
            return [subset] * num_queries
        if len(subset) != num_queries:
            raise ValueError("Subset length must match number of queries.")
        return subset

    def _prepare_search(self, queries_embeddings, subset):
        """fast_plaid.py:743-795"""
        search_indices = self._loaded_indices()
        if not os.path.exists(os.path.join(self.index, "metadata.json")):
            raise FileNotFoundError(
                f"Index metadata not found in '{self.index}'. Please create the index before searching."
            )
        for device in self.devices:
            if device == "cpu":
                raise _engine.EngineUnavailableError(
                    "fast_plaid_b200 has no CPU search path: open the index with device='cuda:N' "
                    "(the CPU restatement of the reference lives in oracle/ and is test-only)."
                )
            if search_indices.get(device) is None:
                raise RuntimeError(
                    f"Index could not be loaded on device '{device}'. Check CUDA memory or device availability."
                )
        queries_embeddings = self._as_query_tensor(queries_embeddings)
        subset = self._per_query_subsets(subset, queries_embeddings.shape[0])
        return search_indices, queries_embeddings, subset

    def _search_device(self, idx: DeviceIndex, queries: torch.Tensor, params,
                       subset: list[list[int]] | None = None) -> list[list[tuple[int, float]]]:
        """search_on_device (fast_plaid.py:188-253) for the whole batch."""
        if queries.dim() != 3:
            raise ValueError(f"Expected a 3D tensor for queries, but got shape {list(queries.shape)}")
        if self.shard is not None:
            return self._search_sharded(idx, queries, params, subset)
        if subset is not None:
            q16 = queries.to(torch.float16).to(idx.device)
            ids, scores, counts = idx.search(q16, params, subset=subset)
            return _results_to_lists(ids.cpu(), scores.cpu(), counts.cpu())
        if queries.device.type == "cuda":
            q16 = queries.to(device=idx.device, dtype=torch.float16)  # fast_plaid.py:241
            ids, scores, counts = idx.search(q16, params)
            return _results_to_lists(ids.cpu(), scores.cpu(), counts.cpu())
        # fp16 cast on the host like the reference (fast_plaid.py:241), straight into pinned staging
        ids, scores, counts = idx.search_host(queries, params)
        return _results_to_lists(ids, scores, counts)

    def _shard_comm(self, idx: DeviceIndex):
        """The NCCL communicator of the sharded search, created on first use (collective: every rank's first
        sharded search creates it).  A world of one needs no process group."""
        if self._comm is None:
            rank, world = self.shard
            if world == 1:
                self._comm = _engine.ShardComm(1, 0, _engine.ShardComm.new_unique_id(), idx.device)
            else:
                self._comm = _engine.ShardComm.from_process_group(idx.device)
        return self._comm

    def _search_sharded(self, idx: DeviceIndex, queries: torch.Tensor, params,
                        subset: list[list[int]] | None = None) -> list[list[tuple[int, float]]]:
        """Document-sharded search: local records -> NCCL all-gather -> global prune + rank."""
        import torch.distributed as dist

        def all_gather(t: torch.Tensor) -> torch.Tensor:
            out = torch.empty((world,) + tuple(t.shape), dtype=t.dtype, device=t.device)
            if world > 1:
                dist.all_gather_into_tensor(out.view(-1), t.contiguous().view(-1))
            else:
                out.copy_(t.unsqueeze(0))
            return out

        rank, world = self.shard
        if subset is None:
            # the whole exchange below the C ABI: one call per batch, both all-gathers on the search stream
            comm = self._shard_comm(idx)
            if queries.device.type == "cpu" and queries.dtype.is_floating_point:
                return _results_to_lists(*idx.search_sharded_host(comm, self.query_groups, queries, params))
            q16 = queries.to(device=idx.device, dtype=torch.float16)
            ids, scores, counts = idx.search_sharded(comm, self.query_groups, q16, params)
            return _results_to_lists(ids.cpu(), scores.cpu(), counts.cpu())
        if self.query_groups != 1:
            raise NotImplementedError("subset= with query_groups > 1: use query_groups=1 (plain document sharding)")
        if queries.device.type == "cpu" and queries.dtype.is_floating_point:
            q16 = idx.stage_queries(queries, params.top_k)  # host cast (fast_plaid.py:241) + async H2D
        else:
            q16 = queries.to(device=idx.device, dtype=torch.float16, non_blocking=True)
        # step 1: local pruning, all-gather of the approximate-score keys
        if subset is None:
            keys = idx.shard_approx_keys(q16, params)
        else:
            # the probe is restricted to the centroids the subset documents touch (search.rs:494-517);
            # with sharded documents that set is the union of the shards' centroid bitmaps
            params = DeviceIndex.with_subset_flag(params)
            cbitmap = idx.shard_subset_begin(q16, params, subset)
            keys = idx.shard_subset_keys(all_gather(cbitmap), int(q16.shape[1]), params)
        all_keys = all_gather(keys)
        # step 2: exact scores of the globally surviving documents only, all-gather of the records
        rec = idx.shard_exact_records(all_keys, rank, int(q16.shape[1]), params)
        ids, scores, counts = idx.merge_records(all_gather(rec), params.top_k)
        return _results_to_lists(ids.cpu(), scores.cpu(), counts.cpu())

    @torch.inference_mode()
    def search(
        self,
        queries_embeddings: torch.Tensor | list[torch.Tensor],
        top_k: int = 10,
        batch_size: int = 2000,
        n_full_scores: int = 4096,
        n_ivf_probe: int = 8,
        show_progress: bool = True,  # noqa: ARG002  (one launch sequence per batch: nothing to show)
        subset: list[list[int]] | list[int] | None = None,
        n_processes: int | None = None,  # noqa: ARG002  (CPU-only knob in the reference)
    ) -> list[list[tuple[int, float]]]:
        """Search the index (fast_plaid.py:930-983).  Returns, per query, up to ``top_k``
        ``(doc_id, score)`` pairs in rank order."""
        search_indices, queries, subset = self._prepare_search(queries_embeddings, subset)
        params = DeviceIndex.make_params(top_k, n_full_scores, n_ivf_probe, batch_size)
        if len(self.devices) == 1:
            return self._search_device(search_indices[self.devices[0]], queries, params, subset)
        # several devices in ONE process: replicated index, query list split across devices
        # (the reference's multi-GPU mode, fast_plaid.py:893-928)
        n = len(self.devices)
        chunk = math.ceil(queries.shape[0] / n)
        chunks = list(torch.split(queries, chunk))
        sub_chunks = [None] * len(chunks) if subset is None else [subset[i : i + chunk] for i in range(0, len(subset), chunk)]
        with ThreadPoolExecutor(max_workers=n) as ex:
            futs = [
                ex.submit(self._search_device, search_indices[d], chunks[i], params, sub_chunks[i])
                for i, d in enumerate(self.devices)
                if i < len(chunks)
            ]
        out: list[list[tuple[int, float]]] = []
        for f in futs:
            out.extend(f.result())
        return out

    @torch.inference_mode()
    def search_token_scores(
        self,
        queries_embeddings: torch.Tensor | list[torch.Tensor],
        top_k: int = 10,
        batch_size: int = 2000,
        n_full_scores: int = 4096,
        n_ivf_probe: int = 8,
        show_progress: bool = True,
        subset: list[list[int]] | list[int] | None = None,
        n_processes: int | None = None,
    ) -> list[list[tuple[int, float, torch.Tensor]]]:
        """``search`` plus, per result, the ``[query_tokens, doc_tokens]`` fp16 similarity
        matrix (fast_plaid.py:985-1043, search.rs:668-686)."""
        base = self.search(queries_embeddings, top_k, batch_size, n_full_scores, n_ivf_probe, show_progress,
                           subset, n_processes)
        search_indices, queries, _ = self._prepare_search(queries_embeddings, None)
        # several devices in one process hold replicas: any of them can produce every matrix
        idx = search_indices[self.devices[0]]
        q16 = queries.to(device=idx.device, dtype=torch.float16)
        pairs_q = torch.tensor([b for b, res in enumerate(base) for _ in res], dtype=torch.int64)
        pairs_d = torch.tensor([d for res in base for d, _ in res], dtype=torch.int64)
        n_pairs = int(pairs_d.shape[0])
        lens_all = (idx.doc_offsets[1:] - idx.doc_offsets[:-1]).cpu()
        if self.shard is None:
            mats = idx.token_scores(q16, pairs_q.to(torch.int32), pairs_d.to(torch.int32))
            lens = lens_all[pairs_d] if n_pairs else torch.zeros(0, dtype=torch.int64)
        else:
            # document-sharded: the rank that holds a document (in the first query group) computes its matrix
            # (search.rs:668-686 on the owning shard); one all-reduce hands every matrix to every rank
            import torch.distributed as dist

            rank, world = self.shard
            group, _, _ = _engine.shard_grid(rank, world, self.query_groups)
            lo, hi = idx.doc_id_base, idx.doc_id_base + idx.num_documents
            own = (pairs_d >= lo) & (pairs_d < hi) & (group == 0)
            own_ix = own.nonzero().flatten()
            mx = torch.tensor([max(idx.max_doc_len, 1)], dtype=torch.int64, device=idx.device)
            if world > 1:
                dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            mats = torch.zeros((max(n_pairs, 1), int(mx), q16.shape[1]), dtype=torch.float16, device=idx.device)
            lens_d = torch.zeros(max(n_pairs, 1), dtype=torch.int64, device=idx.device)
            if own_ix.numel():
                local = idx.token_scores(q16, pairs_q[own_ix].to(torch.int32), (pairs_d[own_ix] - lo).to(torch.int32))
                mats[own_ix.to(idx.device), : local.shape[1]] = local
                lens_d[own_ix.to(idx.device)] = lens_all[pairs_d[own_ix] - lo].to(idx.device)
            if world > 1:
                dist.all_reduce(mats, op=dist.ReduceOp.SUM)  # exactly one rank wrote each matrix, the others hold zeros
                dist.all_reduce(lens_d, op=dist.ReduceOp.SUM)
            lens = lens_d.cpu()
        mats = mats.cpu()
        out, k = [], 0
        for res in base:
            row = []
            for doc_id, score in res:
                n = int(lens[k])
                row.append((doc_id, score, mats[k, :n, :].transpose(0, 1).contiguous()))
                k += 1
            out.append(row)
        return out

    @torch.inference_mode()
    def get_embeddings(self, subset: list[int]) -> list[torch.Tensor]:
        """Decompressed, normalised fp16 embeddings of the given documents
        (fast_plaid.py:1159-1186, embeddings.rs:12-69)."""
        self._check_and_reload_index(blocking=False)
        if not subset:
            return []
        with self._index_swap_lock:
            idx = self.indices.get(self.devices[0])
        if idx is None:
            raise _engine.EngineUnavailableError("get_embeddings needs the index loaded on a CUDA device")
        return [t.cpu() for t in idx.reconstruct(list(subset))]

    # ------------------------------------------------------------------ in-memory construction
    @classmethod
    def from_tensors(cls, data: IndexTensors, device: str, doc_id_base: int = 0) -> DeviceIndex:
        """Bench / test helper: put already-built index tensors straight into HBM."""
        return DeviceIndex(data, device, doc_id_base=doc_id_base)

    @classmethod
    def from_device_index(cls, didx: DeviceIndex, index_dir: str | None = None,
                          shard: tuple[int, int] | None = None, query_groups: int = 1) -> "FastPlaid":
        """A FastPlaid whose index is ALREADY resident in HBM (bench / serving processes that build or receive
        the tensors in memory): `search` runs the same code as for a directory-backed index -- reload check,
        query preparation, C-ABI call, result lists -- the directory only holds the `metadata.json` that check
        looks at."""
        import tempfile

        self = cls.__new__(cls)
        self.devices = [str(didx.device)]
        self.index = index_dir or tempfile.mkdtemp(prefix="fpb_attached_")
        os.makedirs(self.index, exist_ok=True)
        self.low_memory = False
        self.shard = shard
        self.query_groups = int(query_groups)
        self._comm = None
        meta_path = os.path.join(self.index, "metadata.json")
        if not os.path.exists(meta_path):
            with open(meta_path, "w") as f:
                json.dump({"num_documents": didx.num_documents, "nbits": didx.nbits, "attached": True}, f)
        self.lock_path = os.path.join(self.index, "plaid.lock")
        self.lock = FileLock(self.lock_path) if FileLock is not None else _NullLock()
        self._index_swap_lock = threading.Lock()
        self.indices = {self.devices[0]: didx}
        self._cpu_loaded = True
        self._last_known_mtime = Path(meta_path).stat().st_mtime
        return self


def read_num_documents(index_path: str) -> int:
    with open(os.path.join(index_path, "metadata.json")) as f:
        return int(json.load(f).get("num_documents", 0))
