"""ctypes binding of ``libfastplaid_b200.so`` (C ABI in ``include/fastplaid_b200.h``).

This is the only bridge between the Python host and the CUDA kernels.  There is no CPU
fallback: if the shared library is missing or CUDA is unavailable every entry point raises.
PyTorch is used for device memory, streams and (in the sharded mode) ``torch.distributed``.

Reference counterpart: the PyO3 module ``fast_plaid.fast_plaid_rust`` (rust/lib.rs:366-383):
``construct_index`` -> :class:`DeviceIndex`, ``pysearch`` -> :meth:`DeviceIndex.search`.
"""

from __future__ import annotations

import contextlib
import ctypes
import dataclasses
import os
import threading
from typing import Any

import torch

_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc", "libfastplaid_b200.so")
_lib = None
_lib_lock = threading.Lock()

FPB_OK = 0
FPB_ERR_INVALID = -1
FPB_ERR_CUDA = -2
FPB_ERR_UNSUPPORTED = -3
FPB_ERR_WORKSPACE = -4
FPB_ERR_NO_IVF = -5


class EngineUnavailableError(RuntimeError):
    """The CUDA extension is missing or unusable.  There is deliberately no fallback."""


class FpbParams(ctypes.Structure):
    _fields_ = [
        ("n_ivf_probe", ctypes.c_int32),
        ("n_full_scores", ctypes.c_int32),
        ("top_k", ctypes.c_int32),
        ("batch_size", ctypes.c_int32),
        ("flags", ctypes.c_int32),
    ]


FPB_FLAG_SUBSET = 1
FPB_FLAG_APPROX_EXACT_ALL = 2  # off_approx holds the exact score of every candidate (parity tests)
FPB_FLAG_APPROX_DIRECT = 4  # one-pass approximate scoring (A/B alternative of the two-pass default)
FPB_FLAG_APPROX_TWO_PASS = 8  # two passes even for a job the library would score in one (small batch x index)


class FpbLayout(ctypes.Structure):
    _fields_ = [
        ("total_bytes", ctypes.c_int64),
        ("B", ctypes.c_int32),
        ("Q", ctypes.c_int32),
        ("Qp", ctypes.c_int32),
        ("n_tiles", ctypes.c_int32),
        ("R", ctypes.c_int32),
        ("n_probe", ctypes.c_int32),
        ("cand_cap", ctypes.c_int32),
        ("bitmap_words", ctypes.c_int32),
        ("cbitmap_words", ctypes.c_int32),
        ("reserved0", ctypes.c_int32),
        ("off_queries", ctypes.c_int64),
        ("off_S", ctypes.c_int64),
        ("off_tmax", ctypes.c_int64),
        ("off_cells", ctypes.c_int64),
        ("off_bitmap", ctypes.c_int64),
        ("off_n_cand", ctypes.c_int64),
        ("off_cand", ctypes.c_int64),
        ("off_approx", ctypes.c_int64),
        ("off_work", ctypes.c_int64),
        ("off_n_rerank", ctypes.c_int64),
        ("off_rerank", ctypes.c_int64),
        ("off_rerank_approx", ctypes.c_int64),
        ("off_exact", ctypes.c_int64),
        ("off_cbitmap", ctypes.c_int64),
        ("off_clist", ctypes.c_int64),
        ("off_n_clist", ctypes.c_int64),
        ("off_sbitmap", ctypes.c_int64),
        ("off_tau", ctypes.c_int64),
        ("off_hibits", ctypes.c_int64),
        ("off_lb", ctypes.c_int64),
        ("off_refine", ctypes.c_int64),
        ("off_n_refine", ctypes.c_int64),
        ("off_thresh", ctypes.c_int64),
        ("off_work2", ctypes.c_int64),
        ("off_stats", ctypes.c_int64),
        ("hb_words", ctypes.c_int32),
        ("flags", ctypes.c_int32),
    ]


# every symbol include/fastplaid_b200.h declares (checked by tests/test_cabi.py)
EXPORTED_SYMBOLS = [
    "fpb_last_error",
    "fpb_abi_version",
    "fpb_index_create",
    "fpb_index_destroy",
    "fpb_workspace_layout",
    "fpb_search_batch",
    "fpb_search_batch_subset",
    "fpb_search_batch_host",
    "fpb_stage_centroid_scores",
    "fpb_stage_subset",
    "fpb_stage_probe",
    "fpb_stage_candidates",
    "fpb_stage_approx",
    "fpb_stage_select",
    "fpb_stage_maxsim",
    "fpb_stage_rank",
    "fpb_stage_keys",
    "fpb_stage_records",
    "fpb_search_shard",
    "fpb_merge_shards",
    "fpb_shard_approx_keys",
    "fpb_shard_subset_begin",
    "fpb_shard_subset_keys",
    "fpb_shard_apply_threshold",
    "fpb_shard_exact_records",
    "fpb_comm_unique_id",
    "fpb_comm_create",
    "fpb_comm_destroy",
    "fpb_comm_nccl_version",
    "fpb_sharded_scratch_bytes",
    "fpb_search_batch_sharded",
    "fpb_search_batch_sharded_host",
    "fpb_reconstruct",
    "fpb_token_scores",
    "fpb_encode",
    "fpb_kmeans_assign",
    "fpb_kmeans_update",
    "fpb_nearest_centroid",
    "fpb_cast_f32_to_f16_host",
    "fpb_cast_f32_to_f16_host_portable",
]


def library_path() -> str:
    return _LIB_PATH


def load_library() -> ctypes.CDLL:
    """dlopen the C-ABI library (no CUDA call is made)."""
    global _lib
    with _lib_lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(_LIB_PATH):
            raise EngineUnavailableError(
                f"{_LIB_PATH} not found. Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                f"or `make -C fast_plaid_b200/csrc`. The engine has no CPU fallback."
            )
        lib = ctypes.CDLL(_LIB_PATH)
        vp, i32, i64, sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_size_t
        lib.fpb_last_error.restype = ctypes.c_char_p
        lib.fpb_last_error.argtypes = []
        lib.fpb_abi_version.restype = i32
        lib.fpb_index_create.restype = i32
        lib.fpb_index_create.argtypes = [
            ctypes.POINTER(vp), i32, i32, i32, i64, vp, vp, i64, vp, vp, vp, vp, vp, vp, i64, i64, i64,
        ]
        lib.fpb_index_destroy.restype = None
        lib.fpb_index_destroy.argtypes = [vp]
        lib.fpb_workspace_layout.restype = i32
        lib.fpb_workspace_layout.argtypes = [vp, i32, i32, ctypes.POINTER(FpbParams), ctypes.POINTER(FpbLayout)]
        lib.fpb_search_batch.restype = i32
        lib.fpb_search_batch.argtypes = [vp, vp, i32, i32, ctypes.POINTER(FpbParams), vp, sz, vp, vp, vp, vp]
        lib.fpb_search_batch_subset.restype = i32
        lib.fpb_search_batch_subset.argtypes = [vp, vp, i32, i32, ctypes.POINTER(FpbParams), vp, vp, i64, vp, sz,
                                                vp, vp, vp, vp]
        lib.fpb_stage_subset.restype = i32
        lib.fpb_stage_subset.argtypes = [vp, vp, vp, i64, i32, i32, ctypes.POINTER(FpbParams), vp, sz, vp]
        lib.fpb_search_batch_host.restype = i32
        lib.fpb_search_batch_host.argtypes = [
            vp, vp, i32, i32, ctypes.POINTER(FpbParams), vp, sz, vp, vp, vp, vp, vp, vp, vp, vp,
        ]
        lib.fpb_stage_centroid_scores.restype = i32
        lib.fpb_stage_centroid_scores.argtypes = [vp, vp, i32, i32, ctypes.POINTER(FpbParams), vp, sz, vp]
        for name in ("fpb_stage_probe", "fpb_stage_candidates", "fpb_stage_approx", "fpb_stage_select",
                     "fpb_stage_maxsim"):
            fn = getattr(lib, name)
            fn.restype = i32
            fn.argtypes = [vp, i32, i32, ctypes.POINTER(FpbParams), vp, sz, vp]
        lib.fpb_stage_rank.restype = i32
        lib.fpb_stage_rank.argtypes = [vp, i32, i32, ctypes.POINTER(FpbParams), vp, sz, vp, vp, vp, vp]
        lib.fpb_stage_keys.restype = i32
        lib.fpb_stage_keys.argtypes = [vp, i32, i32, ctypes.POINTER(FpbParams), vp, sz, vp, vp]
        lib.fpb_stage_records.restype = i32
        lib.fpb_stage_records.argtypes = [vp, i32, i32, ctypes.POINTER(FpbParams), vp, sz, vp, vp]
        lib.fpb_search_shard.restype = i32
        lib.fpb_search_shard.argtypes = [vp, vp, i32, i32, ctypes.POINTER(FpbParams), vp, sz, vp, vp]
        lib.fpb_shard_approx_keys.restype = i32
        lib.fpb_shard_approx_keys.argtypes = [vp, vp, i32, i32, ctypes.POINTER(FpbParams), vp, sz, vp, vp]
        lib.fpb_shard_subset_begin.restype = i32
        lib.fpb_shard_subset_begin.argtypes = [vp, vp, i32, i32, ctypes.POINTER(FpbParams), vp, vp, i64, vp, sz, vp, vp]
        lib.fpb_shard_subset_keys.restype = i32
        lib.fpb_shard_subset_keys.argtypes = [vp, i32, i32, ctypes.POINTER(FpbParams), vp, sz, vp, i32, vp, vp]
        lib.fpb_shard_apply_threshold.restype = i32
        lib.fpb_shard_apply_threshold.argtypes = [vp, vp, i32, i32, i32, i32, ctypes.POINTER(FpbParams), vp, sz, vp]
        lib.fpb_shard_exact_records.restype = i32
        lib.fpb_shard_exact_records.argtypes = [vp, i32, i32, ctypes.POINTER(FpbParams), vp, sz, vp, vp]
        lib.fpb_comm_unique_id.restype = i32
        lib.fpb_comm_unique_id.argtypes = [vp]
        lib.fpb_comm_create.restype = i32
        lib.fpb_comm_create.argtypes = [ctypes.POINTER(vp), i32, i32, vp, i32]
        lib.fpb_comm_destroy.restype = None
        lib.fpb_comm_destroy.argtypes = [vp]
        lib.fpb_comm_nccl_version.restype = i32
        lib.fpb_sharded_scratch_bytes.restype = i64
        lib.fpb_sharded_scratch_bytes.argtypes = [i32, i32, i32]
        lib.fpb_search_batch_sharded.restype = i32
        lib.fpb_search_batch_sharded.argtypes = [vp, vp, i32, vp, i32, i32, ctypes.POINTER(FpbParams), vp, sz, vp, sz,
                                                 vp, vp, vp, vp]
        lib.fpb_search_batch_sharded_host.restype = i32
        lib.fpb_search_batch_sharded_host.argtypes = [vp, vp, i32, vp, i32, i32, ctypes.POINTER(FpbParams), vp, sz, vp,
                                                      sz, vp, vp, vp, vp, vp, vp, vp, vp]
        lib.fpb_merge_shards.restype = i32
        lib.fpb_merge_shards.argtypes = [vp, i32, i32, i32, i32, vp, vp, vp, vp]
        lib.fpb_reconstruct.restype = i32
        lib.fpb_reconstruct.argtypes = [vp, vp, i32, vp, vp, vp]
        for name in ("fpb_cast_f32_to_f16_host", "fpb_cast_f32_to_f16_host_portable"):
            fn = getattr(lib, name)
            fn.restype = i32
            fn.argtypes = [vp, vp, sz]
        lib.fpb_encode.restype = i32
        lib.fpb_encode.argtypes = [i32, i32, i32, i64, vp, vp, i64, vp, vp, vp, vp]
        lib.fpb_kmeans_assign.restype = i32
        lib.fpb_kmeans_assign.argtypes = [i32, i32, i64, vp, vp, vp, i64, vp, vp]
        lib.fpb_kmeans_update.restype = i32
        lib.fpb_kmeans_update.argtypes = [i32, i32, i64, vp, vp, vp, vp, vp, vp]
        lib.fpb_nearest_centroid.restype = i32
        lib.fpb_nearest_centroid.argtypes = [i32, i32, i64, vp, vp, vp, i64, vp, vp, vp]
        lib.fpb_token_scores.restype = i32
        lib.fpb_token_scores.argtypes = [vp, vp, i32, vp, vp, i32, i64, vp, vp]
        _lib = lib
        return lib


def _check(rc: int) -> None:
    if rc == FPB_OK:
        return
    msg = load_library().fpb_last_error().decode("utf-8", "replace")
    if rc in (FPB_ERR_INVALID, FPB_ERR_NO_IVF, FPB_ERR_UNSUPPORTED):
        raise ValueError(msg)  # anyhow -> PyValueError in the reference (rust/utils/errors.rs:5-7)
    raise RuntimeError(msg)


def _require_cuda() -> None:
    if not torch.cuda.is_available():
        raise EngineUnavailableError(
            "fast_plaid_b200 needs a CUDA device (B200, sm_100a); there is no CPU search path."
        )


def check_supported(dim: int, nbits: int) -> None:
    """The engine's compiled limits (csrc/index.cu fpb_index_create): raise before an index is written."""
    if int(nbits) not in (2, 4):
        raise ValueError(f"unsupported nbits={nbits}: the B200 engine supports nbits 2 and 4")
    if int(dim) not in (64, 128):
        raise ValueError(f"unsupported embedding dim={dim}: the B200 engine supports dim 64 and 128")


def _ptr(t: torch.Tensor | None) -> int | None:
    return None if t is None else t.data_ptr()


@dataclasses.dataclass
class IndexTensors:
    """The immutable tensors of one index (or one document shard), any device.

    Mirrors what ``construct_index`` receives (rust/search/load.rs:122-186).  ``doc_codes``
    may be int64 (on-disk dtype) or int32; ``ivf`` likewise.
    """

    nbits: int
    centroids: torch.Tensor  # [K, D] float
    bucket_weights: torch.Tensor  # [2**nbits]
    doc_lengths: torch.Tensor  # [N] int
    doc_codes: torch.Tensor  # [E] int
    doc_residuals: torch.Tensor  # [E, D*nbits/8] uint8
    ivf: torch.Tensor | None  # [n_ivf] int (doc ids, ascending within a list)
    ivf_lengths: torch.Tensor | None  # [K] int
    avg_residual: torch.Tensor | None = None  # unused at search time (load.rs:146)
    bucket_cutoffs: torch.Tensor | None = None  # unused at search time (load.rs:148)

    @property
    def num_documents(self) -> int:
        return int(self.doc_lengths.shape[0])

    @property
    def dim(self) -> int:
        return int(self.centroids.shape[1])


def encode_tokens(tokens: torch.Tensor, centroids: torch.Tensor, cutoffs: torch.Tensor,
                  nbits: int) -> tuple[torch.Tensor, torch.Tensor]:
    """Index-build encode step on the GPU (fpb_encode; create.rs:404-428): fp16 CUDA tokens [n, 128],
    fp16 centroids [K, 128], f32 cutoffs -> (codes int32 [n], packed residuals u8 [n, 128*nbits/8])."""
    _require_cuda()
    lib = load_library()
    dev = tokens.device
    tokens = tokens.to(torch.float16).contiguous()
    centroids = centroids.to(dev, torch.float16).contiguous()
    cutoffs = cutoffs.to(dev, torch.float32).contiguous()
    n, dim = tokens.shape
    codes = torch.empty((n,), dtype=torch.int32, device=dev)
    res = torch.empty((n, dim * nbits // 8), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _check(lib.fpb_encode(dev.index, int(nbits), int(dim), int(centroids.shape[0]), centroids.data_ptr(),
                              tokens.data_ptr(), n, cutoffs.data_ptr(), codes.data_ptr(), res.data_ptr(),
                              torch.cuda.current_stream(dev).cuda_stream))
    return codes, res


def kmeans_assign(points: torch.Tensor, centroids: torch.Tensor) -> torch.Tensor:
    """Nearest centroid (squared distance) of every fp16 CUDA point [n, 128]: int32 [n] (fpb_kmeans_assign)."""
    _require_cuda()
    lib = load_library()
    dev = points.device
    points = points.to(torch.float16).contiguous()
    centroids = centroids.to(dev, torch.float16).contiguous()
    bias = (-0.5 * (centroids.float() ** 2).sum(1)).contiguous()
    out = torch.empty((points.shape[0],), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _check(lib.fpb_kmeans_assign(dev.index, int(points.shape[1]), int(centroids.shape[0]), centroids.data_ptr(),
                                     bias.data_ptr(), points.data_ptr(), int(points.shape[0]), out.data_ptr(),
                                     torch.cuda.current_stream(dev).cuda_stream))
    return out


def nearest_centroid(points: torch.Tensor, centroids: torch.Tensor,
                     chunk: int = 4_000_000) -> tuple[torch.Tensor, torch.Tensor]:
    """Nearest centroid and squared distance to it of every point [n, 128] (fpb_nearest_centroid; the outlier search
    of update_centroids, update.py:121-150): (assign int32 [n], min_dist2 f32 [n]) on the centroids' CUDA device.

    The points are taken as fp16; min_dist2 = |x|^2 - 2 max_k (<x, c_k> - |c_k|^2 / 2) with |x|^2 summed in fp32 from
    the fp16 point and the dot products accumulated in fp32 on the tensor cores.  Host-resident points are streamed
    to the device `chunk` rows at a time."""
    _require_cuda()
    lib = load_library()
    dev = centroids.device
    if dev.type != "cuda":
        raise ValueError("nearest_centroid: the centroids must be on a CUDA device")
    centroids = centroids.to(torch.float16).contiguous()
    bias = (-0.5 * (centroids.float() ** 2).sum(1)).contiguous()
    n, dim = int(points.shape[0]), int(points.shape[1])
    assign = torch.empty((n,), dtype=torch.int32, device=dev)
    dist2 = torch.empty((n,), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        for s in range(0, n, chunk):
            x = points[s : s + chunk].to(device=dev, dtype=torch.float16).contiguous()
            m = int(x.shape[0])
            best = dist2[s : s + m]
            _check(lib.fpb_nearest_centroid(dev.index, dim, int(centroids.shape[0]), centroids.data_ptr(),
                                            bias.data_ptr(), x.data_ptr(), m, assign[s : s + m].data_ptr(),
                                            best.data_ptr(), stream))
            best.mul_(-2.0).add_((x.float() ** 2).sum(1))
    return assign, dist2


def kmeans_update(points: torch.Tensor, assign: torch.Tensor, centroids: torch.Tensor) -> tuple[torch.Tensor, torch.Tensor]:
    """In-place mean update of `centroids` (fp16 CUDA [K, 128]) from the assignment; returns (counts int64 [K],
    shift f32 [K] = |new - old| of the non-empty clusters, 0 elsewhere).  Deterministic: the points of a cluster
    are summed in index order (fpb_kmeans_update)."""
    _require_cuda()
    lib = load_library()
    dev = points.device
    K = int(centroids.shape[0])
    order = torch.argsort(assign.to(torch.int64), stable=True)
    counts = torch.bincount(assign.to(torch.int64), minlength=K)
    seg = torch.zeros(K + 1, dtype=torch.int64, device=dev)
    seg[1:] = counts.cumsum(0)
    shift = torch.zeros(K, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _check(lib.fpb_kmeans_update(dev.index, int(points.shape[1]), K, points.data_ptr(), order.data_ptr(),
                                     seg.data_ptr(), centroids.data_ptr(), shift.data_ptr(),
                                     torch.cuda.current_stream(dev).cuda_stream))
    return counts, shift


def shard_tensors(data: IndexTensors, rank: int, world: int) -> tuple[IndexTensors, int]:
    """Contiguous document-range shard ``rank`` of ``world`` (SURVEY.md 8e).

    Centroids and bucket weights are replicated; codes/residual rows are a contiguous slice;
    the IVF is rebuilt for the local id range (lists stay ascending because the global lists
    are ascending, create.rs:118-124).  Returns (shard, doc_id_base).
    """
    n = data.num_documents
    lo = (n * rank) // world
    hi = (n * (rank + 1)) // world
    lens = data.doc_lengths.to(torch.int64).cpu()
    offs = torch.cat([torch.zeros(1, dtype=torch.int64), lens.cumsum(0)])
    t0, t1 = int(offs[lo]), int(offs[hi])
    ivf = ivf_lengths = None
    if data.ivf is not None:
        g_ivf = data.ivf.to(torch.int64).cpu()
        g_len = data.ivf_lengths.to(torch.int64).cpu()
        cell_of = torch.repeat_interleave(torch.arange(g_len.shape[0], dtype=torch.int64), g_len)
        keep = (g_ivf >= lo) & (g_ivf < hi)
        ivf = (g_ivf[keep] - lo).to(torch.int32)
        ivf_lengths = torch.bincount(cell_of[keep], minlength=g_len.shape[0]).to(torch.int64)
    shard = IndexTensors(
        nbits=data.nbits,
        centroids=data.centroids,
        bucket_weights=data.bucket_weights,
        doc_lengths=lens[lo:hi],
        doc_codes=data.doc_codes[t0:t1],
        doc_residuals=data.doc_residuals[t0:t1],
        ivf=ivf,
        ivf_lengths=ivf_lengths,
    )
    return shard, lo


# Host -> device upload of the big index arrays (SURVEY 8(f)-2, the loader fast path; the reference goes
# through pageable `.to(device)` copies after materialising int64 codes, load.py:35-322).  Arrays above
# UPLOAD_DIRECT_BYTES are streamed through two pinned staging buffers: the CPU pass that narrows the
# dtype (int64 codes -> int32) writes straight into pinned memory while the previous chunk's DMA runs.
UPLOAD_DIRECT_BYTES = 256 << 20
UPLOAD_CHUNK_BYTES = 64 << 20


def upload_narrow(src: torch.Tensor, device: torch.device, dtype: torch.dtype,
                  out: torch.Tensor | None = None) -> torch.Tensor:
    """src (host, any integer/float dtype, contiguous in dim 0) -> device tensor of `dtype` (`out`, a device tensor
    of the same shape, or a new one).  `src` may be a view of a memory-mapped .npy file: the staging pass is then
    also the disk read."""
    src = src if src.is_contiguous() else src.contiguous()
    out_bytes = src.numel() * torch.empty((), dtype=dtype).element_size()
    if src.device.type != "cpu" or out_bytes <= UPLOAD_DIRECT_BYTES or src.dim() == 0 or src.shape[0] == 0:
        if out is None:
            return src.to(device, dtype).contiguous()
        out.copy_(src.to(dtype) if src.device.type == "cpu" else src)
        return out
    if out is None:
        out = torch.empty(src.shape, dtype=dtype, device=device)
    row_bytes = max(1, out_bytes // src.shape[0])
    rows = max(1, UPLOAD_CHUNK_BYTES // row_bytes)
    stage = [torch.empty((rows,) + tuple(src.shape[1:]), dtype=dtype).pin_memory() for _ in range(2)]
    done = [torch.cuda.Event(), torch.cuda.Event()]
    copy_stream = torch.cuda.Stream(device=device)
    with torch.cuda.stream(copy_stream):
        for i, r0 in enumerate(range(0, src.shape[0], rows)):
            r1 = min(src.shape[0], r0 + rows)
            slot = i & 1
            if i >= 2:
                done[slot].synchronize()  # the DMA that last read this staging buffer has finished
            stage[slot][: r1 - r0].copy_(src[r0:r1])  # dtype narrowing + copy into pinned memory, one pass
            out[r0:r1].copy_(stage[slot][: r1 - r0], non_blocking=True)
            done[slot].record(copy_stream)
    copy_stream.synchronize()
    return out


FPB_COMM_ID_BYTES = 128


class ShardComm:
    """One NCCL communicator created below the C ABI (fpb_comm_*), used by the document-sharded search.

    `ShardComm.from_process_group(device)` bootstraps it from an initialised torch.distributed group: rank 0
    makes the id, the 128 bytes travel through the group's own broadcast (any backend), every rank joins.
    `n_query_groups` x (world / n_query_groups) document shards is the search grid (csrc/comm.cu)."""

    def __init__(self, nranks: int, rank: int, unique_id: bytes, device: torch.device | str) -> None:
        _require_cuda()
        self._lib = load_library()
        self.device = torch.device(device)
        self.nranks, self.rank = int(nranks), int(rank)
        if len(unique_id) != FPB_COMM_ID_BYTES:
            raise ValueError("unique_id must be FPB_COMM_ID_BYTES bytes")
        buf = ctypes.create_string_buffer(bytes(unique_id), FPB_COMM_ID_BYTES)
        handle = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            _check(self._lib.fpb_comm_create(ctypes.byref(handle), self.nranks, self.rank, buf, self.device.index))
        self._handle = handle

    @staticmethod
    def new_unique_id() -> bytes:
        buf = ctypes.create_string_buffer(FPB_COMM_ID_BYTES)
        _check(load_library().fpb_comm_unique_id(buf))
        return buf.raw

    @classmethod
    def from_process_group(cls, device: torch.device | str) -> "ShardComm":
        import torch.distributed as dist

        rank, world = dist.get_rank(), dist.get_world_size()
        box = [cls.new_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        return cls(world, rank, box[0], device)

    def close(self) -> None:
        if getattr(self, "_handle", None) is not None and self._handle.value:
            self._lib.fpb_comm_destroy(self._handle)
            self._handle = ctypes.c_void_p()

    def __del__(self) -> None:  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass


def shard_grid(rank: int, world: int, n_query_groups: int) -> tuple[int, int, int]:
    """(query group, document shard, document shards per group) of `rank` on the n_query_groups x n_shards grid
    of csrc/comm.cu."""
    if n_query_groups < 1 or world % n_query_groups != 0:
        raise ValueError(f"{n_query_groups} query groups do not divide {world} ranks")
    n_shards = world // n_query_groups
    return rank // n_shards, rank % n_shards, n_shards


class DeviceIndex:
    """One index (or shard) resident in HBM + its ``fpb_index`` handle."""

    def __init__(self, data: IndexTensors, device: str | torch.device, doc_id_base: int = 0) -> None:
        _require_cuda()
        self._lib = load_library()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise ValueError(f"Unsupported device string: '{device}' (the B200 engine runs on CUDA only)")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        dev = self.device
        self.nbits = int(data.nbits)
        self.dim = data.dim
        self.doc_id_base = int(doc_id_base)
        with torch.cuda.device(dev):
            # codec tensors are cast to fp16 exactly as construct_index does (load.rs:145-152)
            self.centroids = data.centroids.to(dev, torch.float16).contiguous()
            self.bucket_weights = data.bucket_weights.to(dev, torch.float16).contiguous()
            lens = data.doc_lengths.to(torch.int64)
            self.num_documents = int(lens.shape[0])
            self.max_doc_len = int(lens.max()) if self.num_documents > 0 else 0
            offs = torch.zeros(self.num_documents + 1, dtype=torch.int64)
            offs[1:] = lens.cpu().cumsum(0)
            self.num_tokens = int(offs[-1])
            self.doc_offsets = offs.to(dev)
            # rows past the last document (the reference's tail padding, load.py:298-300) are dropped
            self.doc_codes = upload_narrow(data.doc_codes[: self.num_tokens], dev, torch.int32)
            self.doc_residuals = upload_narrow(data.doc_residuals[: self.num_tokens], dev, torch.uint8)
            if self.doc_codes.numel() == 0:
                self.doc_codes = torch.zeros(1, dtype=torch.int32, device=dev)
                self.doc_residuals = torch.zeros((1, self.dim * self.nbits // 8), dtype=torch.uint8, device=dev)
            self.num_centroids = int(self.centroids.shape[0])
            if data.ivf is not None and data.ivf_lengths is not None:
                il = data.ivf_lengths.to(torch.int64).cpu()
                if il.shape[0] < self.num_centroids:
                    il = torch.cat([il, torch.zeros(self.num_centroids - il.shape[0], dtype=torch.int64)])
                io = torch.zeros(il.shape[0] + 1, dtype=torch.int64)
                io[1:] = il.cumsum(0)
                self.ivf_offsets = io.to(dev)
                self.ivf_pids = upload_narrow(data.ivf, dev, torch.int32)
                if self.ivf_pids.numel() == 0:
                    self.ivf_pids = torch.zeros(1, dtype=torch.int32, device=dev)
                n_ivf = int(io[-1])
            else:
                self.ivf_offsets = None
                self.ivf_pids = None
                n_ivf = 0
            # derived at load: the fp16 norm of every decompressed token (2 B/token), filled by fpb_index_create
            self.token_norms = torch.empty(max(self.num_tokens, 1), dtype=torch.float16, device=dev)
            handle = ctypes.c_void_p()
            _check(
                self._lib.fpb_index_create(
                    ctypes.byref(handle), dev.index, self.nbits, self.dim, self.num_centroids,
                    _ptr(self.centroids), _ptr(self.bucket_weights), self.num_documents,
                    _ptr(self.doc_offsets), _ptr(self.doc_codes), _ptr(self.doc_residuals), _ptr(self.token_norms),
                    _ptr(self.ivf_offsets), _ptr(self.ivf_pids), n_ivf, self.max_doc_len, self.doc_id_base,
                )
            )
        self._handle = handle
        self._ws: dict[tuple, FpbLayout] = {}
        self._buf: torch.Tensor | None = None
        self._io: dict[tuple, dict[str, torch.Tensor]] = {}
        self._lock = threading.Lock()
        # One search at a time per DeviceIndex: the workspace and the staging buffers are shared, and ctypes
        # releases the GIL inside the C-ABI call.  (The fpb_index itself is immutable and thread-safe; callers
        # that want concurrent searches on one GPU give each thread its own workspace through the C ABI.)
        self._search_lock = threading.RLock()
        self._last_stream: torch.cuda.Stream | None = None
        # approximate-stage mode of the host-buffer path (results are identical in both; see _adapt_approx_mode)
        self._approx_direct = False
        self._approx_calls = 0
        self._approx_hold = 0

    @contextlib.contextmanager
    def _exclusive(self):
        with self._search_lock:
            if getattr(self, "_handle", None) is None or not self._handle.value:
                raise RuntimeError("this DeviceIndex has been closed")
            st = torch.cuda.current_stream(self.device)
            if self._last_stream is not None and self._last_stream != st:
                st.wait_stream(self._last_stream)  # the previous call's kernels still own the workspace
            self._last_stream = st
            yield

    # -- lifetime ------------------------------------------------------------------------
    def close(self) -> None:
        lock = getattr(self, "_search_lock", None)
        with (lock if lock is not None else contextlib.nullcontext()):  # wait for a search in flight
            if getattr(self, "_handle", None) is not None and self._handle.value:
                try:
                    torch.cuda.synchronize(self.device)  # kernels still reading the index tensors
                except Exception:
                    pass
                self._lib.fpb_index_destroy(self._handle)
                self._handle = ctypes.c_void_p()
            self._ws = {}
            self._buf = None
            self._io = {}

    def __del__(self) -> None:  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    @property
    def has_ivf(self) -> bool:
        return self.ivf_offsets is not None

    # -- helpers -------------------------------------------------------------------------
    @staticmethod
    def make_params(top_k: int, n_full_scores: int, n_ivf_probe: int, batch_size: int = 2000,
                    flags: int = 0) -> FpbParams:
        return FpbParams(int(n_ivf_probe), int(n_full_scores), int(top_k), int(batch_size), int(flags))

    @staticmethod
    def with_flags(params: FpbParams, flags: int) -> FpbParams:
        return FpbParams(params.n_ivf_probe, params.n_full_scores, params.top_k, params.batch_size,
                         params.flags | int(flags))

    @staticmethod
    def with_subset_flag(params: FpbParams) -> FpbParams:
        return FpbParams(params.n_ivf_probe, params.n_full_scores, params.top_k, params.batch_size,
                         params.flags | FPB_FLAG_SUBSET)

    def layout(self, B: int, Q: int, params: FpbParams) -> FpbLayout:
        lay = FpbLayout()
        _check(self._lib.fpb_workspace_layout(self._handle, B, Q, ctypes.byref(params), ctypes.byref(lay)))
        return lay

    def workspace(self, B: int, Q: int, params: FpbParams) -> tuple[torch.Tensor, FpbLayout]:
        """One grow-only device buffer per index, carved up by fpb_workspace_layout."""
        key = (B, Q, params.n_ivf_probe, params.n_full_scores, params.top_k, params.flags)
        with self._lock:
            lay = self._ws.get(key)
            if lay is None:
                lay = self.layout(B, Q, params)
                if len(self._ws) > 64:
                    self._ws.clear()
                self._ws[key] = lay
            need = int(lay.total_bytes)
            if self._buf is None or self._buf.numel() < need:
                self._buf = None
                self._buf = torch.empty(need, dtype=torch.uint8, device=self.device)
            return self._buf, lay

    def max_queries_per_call(self, Q: int, params: FpbParams, budget_bytes: int = 6 << 30) -> int:
        key = ("maxq", Q, params.n_ivf_probe, params.n_full_scores, params.top_k, params.flags, budget_bytes)
        hit = self._ws.get(key)
        if hit is not None:
            return hit
        val = self._max_queries_per_call(Q, params, budget_bytes)
        self._ws[key] = val
        return val

    def _max_queries_per_call(self, Q: int, params: FpbParams, budget_bytes: int) -> int:
        one = self.layout(1, Q, params).total_bytes
        two = self.layout(2, Q, params).total_bytes
        per_q = max(1, two - one)
        return max(1, int((budget_bytes - one) // per_q) + 1)

    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    # -- search --------------------------------------------------------------------------
    def _subset_csr(self, subset: list[list[int]], s: int, e: int) -> tuple[torch.Tensor, torch.Tensor, int]:
        lens = [len(x) for x in subset[s:e]]
        offs = torch.zeros(len(lens) + 1, dtype=torch.int64)
        offs[1:] = torch.tensor(lens, dtype=torch.int64).cumsum(0)
        flat = [i for x in subset[s:e] for i in x]
        ids = torch.tensor(flat if flat else [0], dtype=torch.int64)
        ids = ids.clamp(-1, 2**31 - 1).to(torch.int32)
        return ids.to(self.device), offs.to(self.device), (max(lens) if lens else 0)

    def search(
        self, queries: torch.Tensor, params: FpbParams, subset: list[list[int]] | None = None
    ) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """queries: fp16 [B, Q, D] on this device.  Returns device tensors
        (ids int64 [B, top_k], scores f32 [B, top_k], counts int32 [B]).  Asynchronous.
        `subset`: per query a list of GLOBAL doc ids to restrict the search to
        (search.rs:494-517, :544-547)."""
        if queries.dim() != 3:
            raise ValueError(f"Expected a 3D tensor for queries, but got shape {list(queries.shape)}")
        if queries.dtype != torch.float16 or queries.device != self.device:
            raise ValueError("DeviceIndex.search expects fp16 queries on the index device")
        queries = queries.contiguous()
        B, Q, D = queries.shape
        if D != self.dim:
            raise ValueError(f"query dim {D} != index dim {self.dim}")
        k = params.top_k
        ids = torch.empty((B, k), dtype=torch.int64, device=self.device)
        scores = torch.empty((B, k), dtype=torch.float32, device=self.device)
        counts = torch.empty((B,), dtype=torch.int32, device=self.device)
        if B == 0:
            return ids, scores, counts
        if subset is not None:
            if len(subset) != B:
                raise ValueError("Subset length must match number of queries.")
            params = FpbParams(params.n_ivf_probe, params.n_full_scores, params.top_k, params.batch_size,
                               params.flags | FPB_FLAG_SUBSET)
        step = self.max_queries_per_call(Q, params)
        with self._exclusive(), torch.cuda.device(self.device):
            for s in range(0, B, step):
                e = min(B, s + step)
                buf, lay = self.workspace(e - s, Q, params)
                if subset is None:
                    _check(
                        self._lib.fpb_search_batch(
                            self._handle, queries[s:e].data_ptr(), e - s, Q, ctypes.byref(params), buf.data_ptr(),
                            buf.numel(), ids[s:e].data_ptr(), scores[s:e].data_ptr(), counts[s:e].data_ptr(),
                            self._stream(),
                        )
                    )
                else:
                    sid, soff, smax = self._subset_csr(subset, s, e)
                    _check(
                        self._lib.fpb_search_batch_subset(
                            self._handle, queries[s:e].data_ptr(), e - s, Q, ctypes.byref(params), sid.data_ptr(),
                            soff.data_ptr(), smax, buf.data_ptr(), buf.numel(), ids[s:e].data_ptr(),
                            scores[s:e].data_ptr(), counts[s:e].data_ptr(), self._stream(),
                        )
                    )
                    self._keepalive = (sid, soff)  # until the stream has consumed them
        return ids, scores, counts

    def _host_io(self, B: int, Q: int, k: int) -> dict[str, torch.Tensor]:
        """Cached pinned + device staging buffers of the host-buffer path."""
        key = (B, Q, k)
        with self._lock:
            io = self._io.get(key)
            if io is None:
                while len(self._io) >= 4:  # a few shapes stay cached (pinning memory costs milliseconds)
                    self._io.pop(next(iter(self._io)))
                D = self.dim
                io = {
                    "d_q": torch.empty((B, Q, D), dtype=torch.float16, device=self.device),
                    "d_ids": torch.empty((B, k), dtype=torch.int64, device=self.device),
                    "d_scores": torch.empty((B, k), dtype=torch.float32, device=self.device),
                    "d_counts": torch.empty((B,), dtype=torch.int32, device=self.device),
                    "h_q": torch.empty((B, Q, D), dtype=torch.float16).pin_memory(),
                    "h_ids": torch.empty((B, k), dtype=torch.int64).pin_memory(),
                    "h_scores": torch.empty((B, k), dtype=torch.float32).pin_memory(),
                    "h_counts": torch.empty((B,), dtype=torch.int32).pin_memory(),
                }
                self._io[key] = io
        return io

    def _cast_into_pinned(self, queries_host: torch.Tensor, h_q: torch.Tensor) -> None:
        """fp32 -> fp16 on the host like the reference (fast_plaid.py:241), straight into pinned memory."""
        if queries_host.dtype == torch.float32 and queries_host.is_contiguous():
            # single-threaded F16C cast in the library: no dependence on ATen's intra-op pool (csrc/host_cast.cu)
            _check(self._lib.fpb_cast_f32_to_f16_host(queries_host.data_ptr(), h_q.data_ptr(), queries_host.numel()))
        else:
            h_q.copy_(queries_host)

    def stage_queries(self, queries_host: torch.Tensor, top_k: int) -> torch.Tensor:
        """Host queries [B, Q, D] -> fp16 device tensor (cached buffer; asynchronous on the current stream)."""
        B, Q, _ = queries_host.shape
        io = self._host_io(B, Q, top_k)
        self._cast_into_pinned(queries_host, io["h_q"])
        io["d_q"].copy_(io["h_q"], non_blocking=True)
        return io["d_q"]

    def search_host(
        self, queries_host: torch.Tensor, params: FpbParams
    ) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """queries_host: float [B, Q, D] in HOST memory.  The H2D copy, the search and the D2H copies of the
        results all happen inside the C-ABI call, which synchronises the stream.  Returns HOST tensors
        (ids, scores, counts)."""
        if queries_host.dim() != 3:
            raise ValueError(f"Expected a 3D tensor for queries, but got shape {list(queries_host.shape)}")
        if queries_host.device.type != "cpu" or not queries_host.dtype.is_floating_point:
            raise ValueError("search_host expects floating-point queries in host memory")
        B, Q, D = queries_host.shape
        if D != self.dim:
            raise ValueError(f"query dim {D} != index dim {self.dim}")
        if B == 0:
            k = params.top_k
            return (torch.empty((0, k), dtype=torch.int64), torch.empty((0, k), dtype=torch.float32),
                    torch.empty((0,), dtype=torch.int32))
        with self._exclusive(), torch.cuda.device(self.device):
            params = self._approx_flags(params)
            step = self.max_queries_per_call(Q, params)
            io = self._host_io(B, Q, params.top_k)
            self._cast_into_pinned(queries_host, io["h_q"])
            queries_host = io["h_q"]
            for s in range(0, B, step):
                e = min(B, s + step)
                buf, lay = self.workspace(e - s, Q, params)
                _check(
                    self._lib.fpb_search_batch_host(
                        self._handle, queries_host[s:e].data_ptr(), e - s, Q, ctypes.byref(params),
                        buf.data_ptr(), buf.numel(), io["d_q"][s:e].data_ptr(), io["d_ids"][s:e].data_ptr(),
                        io["d_scores"][s:e].data_ptr(), io["d_counts"][s:e].data_ptr(),
                        io["h_ids"][s:e].data_ptr(), io["h_scores"][s:e].data_ptr(),
                        io["h_counts"][s:e].data_ptr(), self._stream(),
                    )
                )
            self._adapt_approx_mode(buf, lay)
            # the pinned result buffers are reused by the next call of this shape: hand out copies (77 KB at
            # 64 x 100) while this call still owns them
            return io["h_ids"].clone(), io["h_scores"].clone(), io["h_counts"].clone()

    def search_records(self, queries: torch.Tensor, params: FpbParams) -> torch.Tensor:
        """Sharded mode, local half: returns uint8 [B, R, 16] records (approx f32, exact f32,
        global doc id i64) for this shard's n_full_scores/4 best candidates per query."""
        queries = queries.contiguous()
        B, Q, _ = queries.shape
        buf, lay = self.workspace(B, Q, params)
        rec = torch.empty((B, lay.R, 16), dtype=torch.uint8, device=self.device)
        with self._exclusive(), torch.cuda.device(self.device):
            _check(
                self._lib.fpb_search_shard(
                    self._handle, queries.data_ptr(), B, Q, ctypes.byref(params), buf.data_ptr(), buf.numel(),
                    rec.data_ptr(), self._stream(),
                )
            )
        return rec

    # -- approximate-stage mode --------------------------------------------------------------
    # The two-pass approximate stage (bound pass + exact pass, csrc/k3_approx.cu) wins when most candidates can be
    # discarded by their upper bound (uniform codes: < 1 % re-scored) and loses its fixed costs when the candidates
    # of a query all score alike (strongly clustered corpora: the exact pass then re-scores most of them).  Both
    # modes give bit-identical results, so the host-buffer path simply looks, every APPROX_PROBE_EVERY calls, at the
    # fraction the exact pass re-scored and holds the one-pass mode for a while when it is high.
    APPROX_PROBE_EVERY = 8
    APPROX_DIRECT_ABOVE = 0.30
    APPROX_HOLD_CALLS = 64

    def _approx_flags(self, params: FpbParams) -> FpbParams:
        if self._approx_direct and not (params.flags & (FPB_FLAG_APPROX_EXACT_ALL | FPB_FLAG_APPROX_DIRECT |
                                                        FPB_FLAG_APPROX_TWO_PASS)):
            return self.with_flags(params, FPB_FLAG_APPROX_DIRECT)
        return params

    def _adapt_approx_mode(self, buf: torch.Tensor, lay: FpbLayout) -> None:
        """Called after a synchronised host-buffer search (the workspace still holds its counters)."""
        if self._approx_direct:
            self._approx_hold -= 1
            if self._approx_hold <= 0:
                self._approx_direct = False  # probe the two-pass mode again
            return
        self._approx_calls += 1
        if self._approx_calls % self.APPROX_PROBE_EVERY or lay.flags & FPB_FLAG_APPROX_DIRECT:
            return
        v = self.views(buf, lay)
        both = torch.stack([v["n_refine"].sum(), v["n_cand"].sum()]).cpu()
        n_ref, n_cand = int(both[0]), int(both[1])
        if n_cand > 0 and n_ref / n_cand > self.APPROX_DIRECT_ABOVE:
            self._approx_direct = True
            self._approx_hold = self.APPROX_HOLD_CALLS

    # the whole sharded search in one C-ABI call (both NCCL all-gathers issued inside, csrc/comm.cu)
    def _sharded_io(self, comm: ShardComm, n_query_groups: int, B: int, Q: int, params: FpbParams):
        b_local = -(-B // n_query_groups)
        buf, lay = self.workspace(b_local, Q, params)
        need = int(self._lib.fpb_sharded_scratch_bytes(b_local, lay.R, comm.nranks))
        if getattr(self, "_scratch", None) is None or self._scratch.numel() < need:
            self._scratch = torch.empty(need, dtype=torch.uint8, device=self.device)
        return buf, self._scratch

    def search_sharded(self, comm: ShardComm, n_query_groups: int, queries: torch.Tensor,
                       params: FpbParams) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """queries: fp16 [B, Q, D] on this device, the SAME batch on every rank of `comm` (collective call).
        Returns device tensors (ids, scores, counts) for all B queries."""
        queries = queries.contiguous()
        B, Q, _ = queries.shape
        k = params.top_k
        ids = torch.empty((B, k), dtype=torch.int64, device=self.device)
        scores = torch.empty((B, k), dtype=torch.float32, device=self.device)
        counts = torch.empty((B,), dtype=torch.int32, device=self.device)
        with self._exclusive(), torch.cuda.device(self.device):
            buf, scratch = self._sharded_io(comm, n_query_groups, B, Q, params)
            _check(self._lib.fpb_search_batch_sharded(
                self._handle, comm._handle, n_query_groups, queries.data_ptr(), B, Q, ctypes.byref(params),
                buf.data_ptr(), buf.numel(), scratch.data_ptr(), scratch.numel(), ids.data_ptr(), scores.data_ptr(),
                counts.data_ptr(), self._stream()))
        return ids, scores, counts

    def search_sharded_host(self, comm: ShardComm, n_query_groups: int, queries_host: torch.Tensor,
                            params: FpbParams) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """Host-buffer form of `search_sharded`: fp32/fp16 queries in HOST memory in, host tensors out."""
        B, Q, D = queries_host.shape
        if D != self.dim:
            raise ValueError(f"query dim {D} != index dim {self.dim}")
        with self._exclusive(), torch.cuda.device(self.device):
            io = self._host_io(B, Q, params.top_k)
            self._cast_into_pinned(queries_host, io["h_q"])
            buf, scratch = self._sharded_io(comm, n_query_groups, B, Q, params)
            _check(self._lib.fpb_search_batch_sharded_host(
                self._handle, comm._handle, n_query_groups, io["h_q"].data_ptr(), B, Q, ctypes.byref(params),
                buf.data_ptr(), buf.numel(), scratch.data_ptr(), scratch.numel(), io["d_q"].data_ptr(),
                io["d_ids"].data_ptr(), io["d_scores"].data_ptr(), io["d_counts"].data_ptr(), io["h_ids"].data_ptr(),
                io["h_scores"].data_ptr(), io["h_counts"].data_ptr(), self._stream()))
            return io["h_ids"].clone(), io["h_scores"].clone(), io["h_counts"].clone()

    # two-step sharded search (exact-scores only the globally surviving documents)
    def shard_approx_keys(self, queries: torch.Tensor, params: FpbParams) -> torch.Tensor:
        queries = queries.contiguous()
        B, Q, _ = queries.shape
        buf, lay = self.workspace(B, Q, params)
        keys = torch.empty((B, lay.R), dtype=torch.int64, device=self.device)
        with self._exclusive(), torch.cuda.device(self.device):
            _check(self._lib.fpb_shard_approx_keys(self._handle, queries.data_ptr(), B, Q, ctypes.byref(params),
                                                   buf.data_ptr(), buf.numel(), keys.data_ptr(), self._stream()))
        return keys

    def shard_subset_begin(self, queries: torch.Tensor, params: FpbParams, subset: list[list[int]]) -> torch.Tensor:
        """Sharded search with a `subset`, step 1a: centroid scores and this shard's bitmaps.  Returns the
        shard's centroid bitmap, int32 [B, cbitmap_words], for the all-gather.  `params.flags` must carry
        FPB_FLAG_SUBSET; `subset` holds GLOBAL document ids."""
        queries = queries.contiguous()
        B, Q, _ = queries.shape
        buf, lay = self.workspace(B, Q, params)
        sid, soff, smax = self._subset_csr(subset, 0, B)
        cb = torch.empty((B, lay.cbitmap_words), dtype=torch.int32, device=self.device)
        with self._exclusive(), torch.cuda.device(self.device):
            _check(self._lib.fpb_shard_subset_begin(self._handle, queries.data_ptr(), B, Q, ctypes.byref(params),
                                                    sid.data_ptr(), soff.data_ptr(), smax, buf.data_ptr(),
                                                    buf.numel(), cb.data_ptr(), self._stream()))
            torch.cuda.current_stream(self.device).synchronize()  # sid/soff are temporaries
        return cb

    def shard_subset_keys(self, all_cbitmaps: torch.Tensor, Q: int, params: FpbParams) -> torch.Tensor:
        """Step 1b: all_cbitmaps int32 [n_shards, B, cbitmap_words] (all-gathered) -> int64 keys [B, R]."""
        n_shards, B, _ = all_cbitmaps.shape
        buf, lay = self.workspace(B, Q, params)
        keys = torch.empty((B, lay.R), dtype=torch.int64, device=self.device)
        with self._exclusive(), torch.cuda.device(self.device):
            _check(self._lib.fpb_shard_subset_keys(self._handle, B, Q, ctypes.byref(params), buf.data_ptr(),
                                                   buf.numel(), all_cbitmaps.contiguous().data_ptr(), n_shards,
                                                   keys.data_ptr(), self._stream()))
        return keys

    def shard_exact_records(self, all_keys: torch.Tensor, rank: int, Q: int, params: FpbParams) -> torch.Tensor:
        """all_keys: int64 [n_shards, B, R] (all-gathered).  Applies the global pruning threshold to
        this shard's list, exact-scores the survivors, returns uint8 [B, R, 16] records."""
        n_shards, B, R = all_keys.shape
        buf, lay = self.workspace(B, Q, params)
        rec = torch.empty((B, R, 16), dtype=torch.uint8, device=self.device)
        with self._exclusive(), torch.cuda.device(self.device):
            _check(self._lib.fpb_shard_apply_threshold(self._handle, all_keys.contiguous().data_ptr(), n_shards, rank,
                                                       B, Q, ctypes.byref(params), buf.data_ptr(), buf.numel(),
                                                       self._stream()))
            _check(self._lib.fpb_shard_exact_records(self._handle, B, Q, ctypes.byref(params), buf.data_ptr(),
                                                     buf.numel(), rec.data_ptr(), self._stream()))
        return rec

    def merge_records(
        self, all_records: torch.Tensor, top_k: int
    ) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """all_records: uint8 [n_shards, B, R, 16] (all-gathered).  Global prune + rank."""
        n_shards, B, R, _ = all_records.shape
        ids = torch.empty((B, top_k), dtype=torch.int64, device=self.device)
        scores = torch.empty((B, top_k), dtype=torch.float32, device=self.device)
        counts = torch.empty((B,), dtype=torch.int32, device=self.device)
        with self._exclusive(), torch.cuda.device(self.device):
            _check(
                self._lib.fpb_merge_shards(
                    all_records.contiguous().data_ptr(), n_shards, B, R, top_k, ids.data_ptr(),
                    scores.data_ptr(), counts.data_ptr(), self._stream(),
                )
            )
        return ids, scores, counts

    # -- stage-level access for the parity tests and the roofline bench -------------------
    def run_stages(self, queries: torch.Tensor, params: FpbParams, upto: str = "rank",
                   subset: list[list[int]] | None = None) -> dict[str, Any]:
        """Run the pipeline stage by stage and return views of every intermediate."""
        order = ["centroid_scores", "probe", "candidates", "approx", "select", "maxsim", "rank"]
        if subset is not None:
            params = FpbParams(params.n_ivf_probe, params.n_full_scores, params.top_k, params.batch_size,
                               params.flags | FPB_FLAG_SUBSET)
            order.insert(1, "subset")
        queries = queries.contiguous()
        B, Q, _ = queries.shape
        buf, lay = self.workspace(B, Q, params)
        st = self._stream()
        p = ctypes.byref(params)
        out: dict[str, Any] = {"layout": lay, "workspace": buf}
        with self._exclusive(), torch.cuda.device(self.device):
            for name in order:
                if name == "centroid_scores":
                    _check(self._lib.fpb_stage_centroid_scores(self._handle, queries.data_ptr(), B, Q, p,
                                                               buf.data_ptr(), buf.numel(), st))
                elif name == "subset":
                    sid, soff, smax = self._subset_csr(subset, 0, B)
                    _check(self._lib.fpb_stage_subset(self._handle, sid.data_ptr(), soff.data_ptr(), smax, B, Q, p,
                                                      buf.data_ptr(), buf.numel(), st))
                    torch.cuda.synchronize(self.device)
                elif name == "rank":
                    k = params.top_k
                    ids = torch.empty((B, k), dtype=torch.int64, device=self.device)
                    scores = torch.empty((B, k), dtype=torch.float32, device=self.device)
                    counts = torch.empty((B,), dtype=torch.int32, device=self.device)
                    _check(self._lib.fpb_stage_rank(self._handle, B, Q, p, buf.data_ptr(), buf.numel(),
                                                    ids.data_ptr(), scores.data_ptr(), counts.data_ptr(), st))
                    out.update(ids=ids, scores=scores, counts=counts)
                else:
                    fn = getattr(self._lib, f"fpb_stage_{name}")
                    _check(fn(self._handle, B, Q, p, buf.data_ptr(), buf.numel(), st))
                if name == upto:
                    break
        out.update(self.views(buf, lay))
        return out

    def stage_fn(self, name: str, queries: torch.Tensor, params: FpbParams):
        """A zero-argument callable that launches one stage on the cached workspace (bench)."""
        queries = queries.contiguous()
        B, Q, _ = queries.shape
        buf, lay = self.workspace(B, Q, params)
        p = ctypes.byref(params)
        st = self._stream()
        if name == "centroid_scores":
            return lambda: _check(self._lib.fpb_stage_centroid_scores(
                self._handle, queries.data_ptr(), B, Q, p, buf.data_ptr(), buf.numel(), st))
        fn = getattr(self._lib, f"fpb_stage_{name}")
        return lambda: _check(fn(self._handle, B, Q, p, buf.data_ptr(), buf.numel(), st))

    def views(self, buf: torch.Tensor, lay: FpbLayout) -> dict[str, torch.Tensor]:
        B, Q, Qp, R = lay.B, lay.Q, lay.Qp, lay.R
        K = self.num_centroids

        def v(off: int, nbytes: int, dtype: torch.dtype, shape: tuple) -> torch.Tensor:
            return buf[off : off + nbytes].view(dtype).view(*shape)

        return {
            "S": v(lay.off_S, B * K * Qp * 2, torch.float16, (B, K, Qp)),
            "tmax": v(lay.off_tmax, B * Qp * lay.n_tiles * 2, torch.float16, (B, Qp, lay.n_tiles)),
            "cells": v(lay.off_cells, B * Q * lay.n_probe * 4, torch.int32, (B, Q, lay.n_probe)),
            "n_cand": v(lay.off_n_cand, B * 4, torch.int32, (B,)),
            "cand": v(lay.off_cand, B * lay.cand_cap * 4, torch.int32, (B, lay.cand_cap)),
            "approx": v(lay.off_approx, B * lay.cand_cap * 4, torch.float32, (B, lay.cand_cap)),
            "n_rerank": v(lay.off_n_rerank, B * 4, torch.int32, (B,)),
            "rerank": v(lay.off_rerank, B * R * 4, torch.int32, (B, R)),
            "rerank_approx": v(lay.off_rerank_approx, B * R * 4, torch.float32, (B, R)),
            "exact": v(lay.off_exact, B * R * 4, torch.float32, (B, R)),
            # two-pass approximate stage (absent with FPB_FLAG_APPROX_DIRECT)
            **({} if lay.flags & FPB_FLAG_APPROX_DIRECT else {
                "tau": v(lay.off_tau, B * Qp * 2, torch.float16, (B, Qp)),
                "hibits": v(lay.off_hibits, B * lay.hb_words * 4, torch.int32, (B, lay.hb_words)),
                "approx_lb": v(lay.off_lb, B * lay.cand_cap * 4, torch.float32, (B, lay.cand_cap)),
                "refine": v(lay.off_refine, B * lay.cand_cap * 4, torch.int32, (B, lay.cand_cap)),
            }),
            "n_refine": v(lay.off_n_refine, B * 4, torch.int32, (B,)),
            "thresh": v(lay.off_thresh, B * 4, torch.float32, (B,)),
            "stats": v(lay.off_stats, 64, torch.int64, (8,)),
        }

    # -- by-products -----------------------------------------------------------------------
    def reconstruct(self, doc_ids: list[int]) -> list[torch.Tensor]:
        """reconstruct_embeddings (rust/utils/embeddings.rs:12-69): fp16 [len, D] per doc."""
        if not doc_ids:
            return []
        ids = torch.tensor(doc_ids, dtype=torch.int64)
        if int(ids.min()) < 0 or int(ids.max()) >= self.num_documents:
            raise ValueError("document id out of range")
        offs = self.doc_offsets.cpu()
        lens = offs[ids + 1] - offs[ids]
        out_off = torch.zeros(len(doc_ids) + 1, dtype=torch.int64)
        out_off[1:] = lens.cumsum(0)
        total = int(out_off[-1])
        out = torch.empty((max(total, 1), self.dim), dtype=torch.float16, device=self.device)
        d_ids = ids.to(self.device, torch.int32)
        d_off = out_off.to(self.device)
        with self._exclusive(), torch.cuda.device(self.device):
            _check(self._lib.fpb_reconstruct(self._handle, d_ids.data_ptr(), len(doc_ids), d_off.data_ptr(),
                                             out.data_ptr(), self._stream()))
        return [out[int(out_off[i]) : int(out_off[i + 1])] for i in range(len(doc_ids))]

    def token_scores(self, queries: torch.Tensor, query_of: torch.Tensor, doc_ids: torch.Tensor) -> torch.Tensor:
        """fp16 [n, max_len, Q] token matrices for explicit (query, local doc) pairs."""
        queries = queries.contiguous()
        n = int(doc_ids.shape[0])
        Q = int(queries.shape[1])
        out = torch.zeros((max(n, 1), max(self.max_doc_len, 1), Q), dtype=torch.float16, device=self.device)
        if n == 0:
            return out[:0]
        qo = query_of.to(self.device, torch.int32).contiguous()
        di = doc_ids.to(self.device, torch.int32).contiguous()
        with self._exclusive(), torch.cuda.device(self.device):
            _check(self._lib.fpb_token_scores(self._handle, queries.data_ptr(), Q, qo.data_ptr(), di.data_ptr(), n,
                                              max(self.max_doc_len, 1), out.data_ptr(), self._stream()))
        return out
