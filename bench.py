#!/usr/bin/env python
"""Benchmark of the PLAID search hot path (BASELINE.json metric: queries/sec @ top_k=100 on a
1M-doc x 300-tok x 128-dim index; MaxSim HBM GB/s vs roofline).

    python bench.py --gpus 1 --steps 5 --warmup 3                # B200 engine (default)
    python bench.py --impl reference --gpus 1 --steps 5 --warmup 3   # the reference's CPU path
    python bench.py --gpus 1 --steps 5 --warmup 3 --dump-outputs DIR   # also write the last step's results
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...   # document-sharded

A "step" is one batch of 64 queries x 32 tokens through the whole hot path.  `value` is
queries/sec with the queries already resident in HBM (stage by stage through the C ABI, CUDA
events between the stages); `e2e` is the same through the user-facing call
`FastPlaid.search(fp32 host queries, top_k=...)` -> `list[list[(doc_id, score)]]`, host<->device
copies inside the timed region.  One JSON line on stdout.

Parity is part of the line: `parity_sample` runs the CPU oracle on the first queries of a batch, at
any number of GPUs, and classifies every difference between the engine's id lists and the oracle's.

`--dump-outputs DIR` writes what the timed path returned in its last step -- DIR/ids.npy (float64 [B, top_k],
-1 past the count), DIR/scores.npy (float32 [B, top_k], -inf past the count), DIR/counts.npy (float64 [B]) --
so that two builds run with the same arguments (hence the same seeded index and queries) can be compared output for
output.
"""

from __future__ import annotations

import argparse
import datetime
import importlib.util
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

CONFIGS = {
    # name: n_docs, doc_len, B, Q, top_k
    "cfg3": dict(n_docs=1_000_000, doc_len=300, B=64, Q=32, top_k=100,
                 desc="1M docs x 300 tok x 128-dim (nbits=4, K=262144), batch=64 queries x 32 tok, top_k=100"),
    "cfg3c": dict(n_docs=1_000_000, doc_len=300, B=64, Q=32, top_k=100, topics=4096, mix=0.05,
                  desc="clustered variant of cfg3: 4096 topics x 64 centroids, 5 % of the codes uniform "
                       "(1M docs x 300 tok, K=262144), batch=64 queries x 32 tok, top_k=100"),
    "cfg2": dict(n_docs=100_000, doc_len=300, B=64, Q=32, top_k=100,
                 desc="100k docs x 300 tok x 128-dim (nbits=4, K=65536), batch=64 queries x 32 tok, top_k=100"),
    "cfg4": dict(n_docs=1_000_000, doc_len=300, B=256, Q=32, top_k=1000,
                 desc="1M docs x 300 tok x 128-dim sharded, batch=256 queries x 32 tok, top_k=1000"),
    "cfg5": dict(n_docs=50_000, doc_len=1024, B=32, Q=64, top_k=10,
                 desc="ColPali shape: 50k docs x 1024 tok x 128-dim, batch=32 queries x 64 tok, top_k=10"),
    "tiny": dict(n_docs=20_000, doc_len=100, B=16, Q=32, top_k=10,
                 desc="20k docs x 100 tok (plumbing check)"),
}
DIM, NBITS, N_IVF_PROBE, N_FULL = 128, 4, 8, 4096
SEED_INDEX, SEED_QUERY = 1234, 4321
N_QUERY_BATCHES = 4  # distinct query batches rotated across steps
PARITY_QUERIES = 16  # queries cross-checked against the oracle (and classified) per run


# ----------------------------------------------------------------------------------------
def measured_peak_hbm() -> tuple[float, str]:
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            with open(p) as f:
                return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int) -> None:
        self.gpu = gpu_index
        self.lines: list[str] = []
        self.proc: subprocess.Popen | None = None
        self.thread: threading.Thread | None = None

    def start(self) -> None:
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return

        def pump():
            for line in self.proc.stdout:  # type: ignore[union-attr]
                self.lines.append(line.strip())

        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
            self.proc.wait()
        if self.thread is not None:
            self.thread.join(timeout=5)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {
            "sm_mhz": statistics.median(sm) if sm else None,
            "sm_max_mhz": max(mx) if mx else None,
            "samples": len(sm),
            "reasons": sorted(reasons),
        }


def dist_setup():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist

        torch.cuda.set_device(local)
        # rank 0 runs the CPU oracle (parity sample) while the others wait at a barrier: generous timeout
        dist.init_process_group("nccl", device_id=torch.device("cuda", local),
                                timeout=datetime.timedelta(minutes=45))
    return rank, world, local


# ----------------------------------------------------------------------------------------
# Synthetic inputs.  Plain torch, shared verbatim by both arms; neither the engine nor the oracle is involved.
def load_synthetic_module():
    """fast_plaid_b200/index/synthetic.py loaded BY FILE PATH: the generator is pure torch, and this keeps the
    package (and every shared library of it) out of the reference arm's process."""
    path = os.path.join(ROOT, "fast_plaid_b200", "index", "synthetic.py")
    spec = importlib.util.spec_from_file_location("_fpb_bench_synthetic", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _bitrev(x: torch.Tensor, nbits: int) -> torch.Tensor:
    r = torch.zeros_like(x)
    for k in range(nbits):
        r |= ((x >> k) & 1) << (nbits - 1 - k)
    return r


def decompressed_tokens(centroids, weights, codes, residuals) -> torch.Tensor:
    """fp32 [n, DIM]: centroid + bucket weight per dimension, L2-normalised.  Only used to MAKE query inputs
    (noisy copies of document tokens); it is a plain-torch statement of the codec, not the engine or the oracle."""
    hi, lo = (residuals >> 4).long(), (residuals & 15).long()  # nbits = 4: two elements per byte, high nibble first
    idx = torch.stack([hi, lo], dim=-1).reshape(residuals.shape[0], -1)
    w = weights.float()[_bitrev(idx, NBITS)]
    e = centroids.float()[codes.long()] + w
    return torch.nn.functional.normalize(e, dim=-1)


def query_source_docs(n_docs: int) -> int:
    """Queries are noisy copies of tokens of documents drawn among the first n_docs/8: inside rank 0's shard for
    every world size of the scaling run, so that every world size (and both arms) searches the same queries."""
    return max(1, n_docs // 8)


def make_query_batches(arrays, n_source_docs: int, cfg, n_batches: int) -> torch.Tensor:
    """fp32 host queries [n_batches, B, Q, D] from (a shard of) the synthetic index on any device."""
    g = torch.Generator().manual_seed(SEED_QUERY)
    B, Q = cfg["B"], cfg["Q"]
    n = n_batches * B
    lens = arrays.doc_lengths[:n_source_docs].to(torch.int64).cpu()
    offs = torch.zeros(lens.shape[0] + 1, dtype=torch.int64)
    offs[1:] = lens.cumsum(0)
    doc_ids = torch.randint(0, n_source_docs, (n,), generator=g).tolist()
    cent, wts = arrays.centroids.cpu(), arrays.bucket_weights.cpu()
    out = torch.empty(n, Q, DIM)
    for i, d in enumerate(doc_ids):
        t0, t1 = int(offs[d]), int(offs[d + 1])
        e = decompressed_tokens(cent, wts, arrays.doc_codes[t0:t1].cpu(), arrays.doc_residuals[t0:t1].cpu())
        rows = torch.randint(0, max(1, e.shape[0]), (Q,), generator=g)
        x = e[rows] + 0.2 * torch.randn(Q, DIM, generator=g)
        out[i] = torch.nn.functional.normalize(x, dim=-1)
    return out.view(n_batches, B, Q, DIM)


# ----------------------------------------------------------------------------------------
def maxsim_algorithmic_bytes(didx, views, lay) -> int:
    """SURVEY.md 8(d): per query T_r*(pd+4) + R*8 + Q*D*2 + R*4, centroid table once per batch."""
    pd = DIM * NBITS // 8
    lens = (didx.doc_offsets[1:] - didx.doc_offsets[:-1])
    total = 0
    n_rr = views["n_rerank"].cpu()
    for b in range(lay.B):
        r = int(n_rr[b])
        ids = views["rerank"][b, :r].long()
        t_r = int(lens[ids].sum()) if r > 0 else 0
        total += t_r * (pd + 4) + r * 8 + lay.Q * DIM * 2 + r * 4
    return total + didx.num_centroids * DIM * 2


def approx_algorithmic_bytes(didx, views, lay) -> tuple[int, int]:
    """HBM bytes (codes + ids + scores) of the approximate stage and its candidate tokens."""
    lens = (didx.doc_offsets[1:] - didx.doc_offsets[:-1])
    hbm = tokens = 0
    n_c = views["n_cand"].cpu()
    for b in range(lay.B):
        n = int(n_c[b])
        ids = views["cand"][b, :n].long()
        t_c = int(lens[ids].sum()) if n > 0 else 0
        hbm += t_c * 4 + n * 12
        tokens += t_c
    return hbm, tokens


def traffic_for(config: str, world: int):
    """ncu dram__bytes_read+write of the MaxSim kernel per launch, from the capture committed for exactly this
    (config, world size); None when there is none."""
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        with open(tp) as f:
            entry = json.load(f).get(f"{config}@{world}")
        return (entry or {}).get("k5_maxsim_dram_bytes_per_launch"), (entry or {}).get("source")
    except Exception:
        return None, None


HBM_INDEX_BUDGET = 60e9  # bytes of one GPU's 180 GB given to index data; the rest is score table, workspace, headroom


def default_query_groups(world: int, cfg: dict) -> int:
    """Grid policy: the FEWEST document shards whose slice fits the per-GPU budget, every other rank a query group.
    Splitting the queries costs nothing (they are independent; each rank runs K1 / the probe on its own B / groups
    queries), splitting the documents repeats those stages on every shard and adds the pruning exchange -- measured
    on cfg3: 2 x 1 beats 1 x 2 by 11 %, 4 x 1 beats 2 x 2 by 6 % (profiles/r02_summary.md).  Documents are sharded
    when the index needs it (or on request: --query-groups)."""
    tokens = cfg["n_docs"] * cfg["doc_len"]
    index_bytes = tokens * (DIM * NBITS // 8 + 4 + 2 + 4)  # residuals, int32 code, fp16 norm, inverted-file entry
    for n_shards in range(1, world + 1):
        if world % n_shards == 0 and index_bytes / n_shards <= HBM_INDEX_BUDGET:
            return world // n_shards
    return 1


# ----------------------------------------------------------------------------------------
def run_b200(args) -> dict:
    from fast_plaid_b200.engine import FPB_FLAG_APPROX_DIRECT, DeviceIndex, IndexTensors, ShardComm, _check, shard_grid
    from fast_plaid_b200.search.fast_plaid import FastPlaid

    rank, world, local = dist_setup()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback in the engine)")
    import torch.distributed as dist

    device = f"cuda:{local}"
    torch.cuda.set_device(local)
    cfg = CONFIGS[args.config]
    n_docs = cfg["n_docs"]
    # the grid of the sharded search: query groups x document shards (csrc/comm.cu)
    n_groups = args.query_groups or default_query_groups(world, cfg)
    group, doc_shard, n_shards = shard_grid(rank, world, n_groups)
    lo, hi = (n_docs * doc_shard) // n_shards, (n_docs * (doc_shard + 1)) // n_shards
    synth = load_synthetic_module()
    t0 = time.time()
    arrays, base = synth.synthetic_arrays(n_docs, cfg["doc_len"], DIM, NBITS, device, SEED_INDEX, doc_range=(lo, hi),
                                          topics=cfg.get("topics", 0), mix=cfg.get("mix", 0.05))
    data = IndexTensors(nbits=arrays.nbits, centroids=arrays.centroids, bucket_weights=arrays.bucket_weights,
                        doc_lengths=arrays.doc_lengths, doc_codes=arrays.doc_codes,
                        doc_residuals=arrays.doc_residuals, ivf=arrays.ivf, ivf_lengths=arrays.ivf_lengths)
    didx = DeviceIndex(data, device, doc_id_base=base)
    torch.cuda.synchronize()
    t_index = time.time() - t0
    params = DeviceIndex.make_params(cfg["top_k"], N_FULL, N_IVF_PROBE)
    if args.approx == "direct":  # A/B: one-pass approximate stage (every row of every candidate gathered)
        params = DeviceIndex.with_flags(params, FPB_FLAG_APPROX_DIRECT)
    B, Q = cfg["B"], cfg["Q"]

    # queries: rank 0 makes them, everybody gets the same ones
    if rank == 0:
        q_host = make_query_batches(arrays, min(query_source_docs(n_docs), hi - lo), cfg, N_QUERY_BATCHES)
    else:
        q_host = torch.empty(N_QUERY_BATCHES, B, Q, DIM)
    del data, arrays
    if world > 1:
        qd = q_host.to(device)
        dist.broadcast(qd, 0)
        q_host = qd.cpu()
    q_host = q_host.pin_memory()
    q_dev16 = q_host.to(device).half()

    lib = didx._lib
    import ctypes

    buf, lay = didx.workspace(B, Q, params)
    pp = ctypes.byref(params)
    st = didx._stream()
    k = params.top_k
    ids = torch.empty((B, k), dtype=torch.int64, device=device)
    scores = torch.empty((B, k), dtype=torch.float32, device=device)
    counts = torch.empty((B,), dtype=torch.int32, device=device)
    rec = torch.empty((B, lay.R, 16), dtype=torch.uint8, device=device)
    gathered = torch.empty((world, B, lay.R, 16), dtype=torch.uint8, device=device)
    keys = torch.empty((B, lay.R), dtype=torch.int64, device=device)
    all_keys = torch.empty((world, B, lay.R), dtype=torch.int64, device=device)
    last = [ids, scores, counts]  # what the timed path returned in its latest step
    stage_names = ["centroid_scores", "probe", "candidates", "approx", "select", "maxsim", "final"]
    if world > 1:
        stage_names = ["centroid_scores", "probe", "candidates", "approx", "select", "exchange_keys", "maxsim", "final"]

    def one_step(qb: torch.Tensor, events: list | None) -> None:
        def mark():
            if events is not None:
                e = torch.cuda.Event(enable_timing=True)
                e.record()
                events.append(e)

        mark()
        _check(lib.fpb_stage_centroid_scores(didx._handle, qb.data_ptr(), B, Q, pp, buf.data_ptr(), buf.numel(), st))
        mark()
        _check(lib.fpb_stage_probe(didx._handle, B, Q, pp, buf.data_ptr(), buf.numel(), st))
        mark()
        _check(lib.fpb_stage_candidates(didx._handle, B, Q, pp, buf.data_ptr(), buf.numel(), st))
        mark()
        _check(lib.fpb_stage_approx(didx._handle, B, Q, pp, buf.data_ptr(), buf.numel(), st))
        mark()
        _check(lib.fpb_stage_select(didx._handle, B, Q, pp, buf.data_ptr(), buf.numel(), st))
        mark()
        if world > 1:
            # two-step sharded search: global pruning threshold before the exact stage
            _check(lib.fpb_stage_keys(didx._handle, B, Q, pp, buf.data_ptr(), buf.numel(), keys.data_ptr(), st))
            dist.all_gather_into_tensor(all_keys.view(-1), keys.view(-1))
            _check(lib.fpb_shard_apply_threshold(didx._handle, all_keys.data_ptr(), world, rank, B, Q, pp,
                                                 buf.data_ptr(), buf.numel(), st))
            mark()
        _check(lib.fpb_stage_maxsim(didx._handle, B, Q, pp, buf.data_ptr(), buf.numel(), st))
        mark()
        if world == 1:
            _check(lib.fpb_stage_rank(didx._handle, B, Q, pp, buf.data_ptr(), buf.numel(), ids.data_ptr(),
                                      scores.data_ptr(), counts.data_ptr(), st))
        else:
            _check(lib.fpb_stage_records(didx._handle, B, Q, pp, buf.data_ptr(), buf.numel(), rec.data_ptr(), st))
            dist.all_gather_into_tensor(gathered.view(-1), rec.view(-1))
            _check(lib.fpb_merge_shards(gathered.data_ptr(), world, B, lay.R, k, ids.data_ptr(), scores.data_ptr(),
                                        counts.data_ptr(), st))
        mark()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    comm = ShardComm.from_process_group(device) if world > 1 else None

    if world > 1:
        # N > 1: the timed step is the product path -- ONE C-ABI call per batch, both ncclAllGather issued inside on
        # the search stream (fpb_search_batch_sharded).  The per-stage table comes from a separate staged pass.
        stage_names = ["whole_call"]

        def one_step(qb: torch.Tensor, events: list | None) -> None:  # noqa: F811
            if events is not None:
                e0 = torch.cuda.Event(enable_timing=True)
                e0.record()
                events.append(e0)
            last[:] = didx.search_sharded(comm, n_groups, qb, params)
            if events is not None:
                e1 = torch.cuda.Event(enable_timing=True)
                e1.record()
                events.append(e1)

    for w in range(args.warmup):
        one_step(q_dev16[w % N_QUERY_BATCHES], None)
    barrier()

    (didx.views(*didx.workspace(-(-B // n_groups), Q, params)) if world > 1 else didx.views(buf, lay))["stats"].zero_()  # approximate-stage counters: timed steps only
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.3)
    all_events: list[list] = []
    barrier()
    t_wall0 = time.time()
    for s in range(args.steps):
        ev: list = []
        one_step(q_dev16[s % N_QUERY_BATCHES], ev)
        all_events.append(ev)
    barrier()
    t_wall = time.time() - t_wall0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last)
    total_ms = all_events[0][0].elapsed_time(all_events[-1][-1])
    stage_ms = [0.0] * len(stage_names)
    for ev in all_events:
        for i in range(len(stage_names)):
            stage_ms[i] += ev[i].elapsed_time(ev[i + 1])
    stage_ms = [x / args.steps for x in stage_ms]
    if world > 1:  # the sharded call lays the workspace out for this rank's slice of the batch
        buf, lay = didx.workspace(-(-B // n_groups), Q, params)
    views = didx.views(buf, lay)
    ms_bytes = maxsim_algorithmic_bytes(didx, views, lay)
    ap_hbm, ap_tokens = approx_algorithmic_bytes(didx, views, lay)
    n_cand_mean = float(views["n_cand"].float().mean())
    k3_stats = [int(x) for x in views["stats"].cpu().tolist()]
    n_refine_mean = float(views["n_refine"].float().mean()) if args.approx != "direct" else None

    # ---- e2e: FastPlaid.search(fp32 host queries) -> Python lists, copies inside the timed region ----
    fp = FastPlaid.from_device_index(didx, shard=(rank, world) if world > 1 else None, query_groups=n_groups)
    fp._comm = comm  # one communicator for the device-timed and the end-to-end legs
    n_full = N_FULL

    def e2e_call(qb_host: torch.Tensor):
        if args.approx == "direct":  # the A/B flag is not part of the FastPlaid surface
            return fp._search_device(didx, qb_host, params)
        return fp.search(qb_host, top_k=k, n_full_scores=n_full, n_ivf_probe=N_IVF_PROBE, show_progress=False)

    for w in range(max(1, min(args.warmup, 2))):
        e2e_call(q_host[w % N_QUERY_BATCHES])
    barrier()
    t0 = time.time()
    for s in range(args.steps):
        res = e2e_call(q_host[s % N_QUERY_BATCHES])
    barrier()
    t_e2e = time.time() - t0
    clocks = sampler.stop()
    assert len(res) == B

    # max over ranks
    tt = torch.tensor([total_ms, t_e2e * 1000.0], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    total_ms, e2e_ms = float(tt[0]), float(tt[1])

    peak, peak_src = measured_peak_hbm()
    if world > 1:
        # stage breakdown of the sharded step: the same sequence once more through the step-wise entry points, the two
        # all-gathers issued through torch.distributed here (the timed product path issues them below the C ABI)
        whole = stage_ms[0]
        b_local = -(-B // n_groups)
        nb = max(0, min(b_local, B - group * b_local))
        stage_names = ["centroid_scores", "probe", "candidates", "approx", "select", "exchange_keys", "maxsim",
                       "exchange_records_and_merge"]
        acc = [0.0] * len(stage_names)
        per_rank = b_local * lay.R
        keys_l = torch.zeros((b_local, lay.R), dtype=torch.int64, device=device)
        keys_all = torch.zeros((world, b_local, lay.R), dtype=torch.int64, device=device)
        rec_l = torch.full((b_local, lay.R, 16), 255, dtype=torch.uint8, device=device)
        rec_all = torch.zeros((world, b_local, lay.R, 16), dtype=torch.uint8, device=device)
        reps = 3
        for rep in range(reps):
            qs = q_dev16[rep % N_QUERY_BATCHES][group * b_local: group * b_local + nb].contiguous()
            bufs, lays = didx.workspace(max(nb, 1), Q, params)
            pl = ctypes.byref(params)
            evs = [torch.cuda.Event(enable_timing=True) for _ in range(len(stage_names) + 1)]
            h = didx._handle
            evs[0].record()
            if nb:
                _check(lib.fpb_stage_centroid_scores(h, qs.data_ptr(), nb, Q, pl, bufs.data_ptr(), bufs.numel(), st))
            evs[1].record()
            if nb:
                _check(lib.fpb_stage_probe(h, nb, Q, pl, bufs.data_ptr(), bufs.numel(), st))
            evs[2].record()
            if nb:
                _check(lib.fpb_stage_candidates(h, nb, Q, pl, bufs.data_ptr(), bufs.numel(), st))
            evs[3].record()
            if nb:
                _check(lib.fpb_stage_approx(h, nb, Q, pl, bufs.data_ptr(), bufs.numel(), st))
            evs[4].record()
            if nb:
                _check(lib.fpb_stage_select(h, nb, Q, pl, bufs.data_ptr(), bufs.numel(), st))
            evs[5].record()
            if nb:
                _check(lib.fpb_stage_keys(h, nb, Q, pl, bufs.data_ptr(), bufs.numel(), keys_l.data_ptr(), st))
            dist.all_gather_into_tensor(keys_all.view(-1), keys_l.view(-1))
            if nb:
                # the kernel strides the gathered keys by the queries per rank (b_local); this rank's group starts at
                # shard 0 of the group
                grp_keys = keys_all[group * n_shards:(group + 1) * n_shards]
                if nb == b_local:
                    _check(lib.fpb_shard_apply_threshold(h, grp_keys.data_ptr(), n_shards, doc_shard, nb, Q, pl,
                                                         bufs.data_ptr(), bufs.numel(), st))
                else:  # ragged last group: repack to the stride the step-wise entry point expects
                    gk = grp_keys[:, :nb].contiguous()
                    _check(lib.fpb_shard_apply_threshold(h, gk.data_ptr(), n_shards, doc_shard, nb, Q, pl,
                                                         bufs.data_ptr(), bufs.numel(), st))
            evs[6].record()
            if nb:
                _check(lib.fpb_stage_maxsim(h, nb, Q, pl, bufs.data_ptr(), bufs.numel(), st))
            evs[7].record()
            if nb:
                _check(lib.fpb_stage_records(h, nb, Q, pl, bufs.data_ptr(), bufs.numel(), rec_l.data_ptr(), st))
            dist.all_gather_into_tensor(rec_all.view(-1), rec_l.view(-1))
            for g in range(n_groups):
                gn = max(0, min(b_local, B - g * b_local))
                if gn == 0:
                    continue
                gr = rec_all[g * n_shards:(g + 1) * n_shards]
                gr = gr if gn == b_local else gr[:, :gn].contiguous()
                _check(lib.fpb_merge_shards(gr.data_ptr(), n_shards, gn, lay.R, k, ids[g * b_local:].data_ptr(),
                                            scores[g * b_local:].data_ptr(), counts[g * b_local:].data_ptr(), st))
            evs[8].record()
            torch.cuda.synchronize()
            if rep > 0:  # the first repetition warms the step-wise path up
                for i in range(len(stage_names)):
                    acc[i] += evs[i].elapsed_time(evs[i + 1])
        stage_ms = [x / (reps - 1) for x in acc]
        if nb:
            buf, lay = didx.workspace(nb, Q, params)
            views = didx.views(buf, lay)
            ms_bytes = maxsim_algorithmic_bytes(didx, views, lay)
            ap_hbm, ap_tokens = approx_algorithmic_bytes(didx, views, lay)
        stage_names.append("whole_call")
        stage_ms.append(whole)
    i_ms = stage_names.index("maxsim")
    i_ap = stage_names.index("approx")
    ms_time = stage_ms[i_ms] / 1000.0
    achieved = ms_bytes / ms_time / 1e9 if ms_time > 0 else 0.0
    traffic, traffic_src = traffic_for(args.config, world)
    h2d = B * Q * DIM * 2
    d2h = B * k * 12 + B * 4
    n_launch = count_launches(world, args.approx)
    out = {
        "metric": "queries/sec @ top_k=%d, %s-doc/128-dim index; MaxSim HBM GB/s vs roofline" % (
            cfg["top_k"], "1M" if n_docs == 1_000_000 else str(n_docs)),
        "value": B * args.steps / (total_ms / 1000.0),
        "unit": "queries/s",
        "n_gpus": world,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": total_ms / args.steps,
        "higher_is_better": True,
        "scaling": "strong",
        "vs_baseline": None,
        "dtype": "f16",
        "data": "synthetic (seeded direct-layout index: normalised random centroids, uniform codes, uniform "
                "residual nibbles; queries = noisy copies of decompressed document tokens)",
        "config": {
            "workload": f"{args.config}: {cfg['desc']}",
            "n_ivf_probe": N_IVF_PROBE, "n_full_scores": N_FULL, "reranked_per_query": lay.R,
            "parallelism": (f"{n_groups} query groups x {n_shards} document shards, both ncclAllGather (approximate-score "
                            "keys, then records of the globally surviving documents) issued below the C ABI"
                            if world > 1 else "one GPU"),
            "l2": "inputs larger than L2: 20 GB index, 1.07 GB score table per batch; "
                  f"{N_QUERY_BATCHES} distinct query batches rotate across steps",
            "candidates_per_query_mean": n_cand_mean,
            "index_build_s": round(t_index, 1),
        },
        "e2e": {"value": B * args.steps / (e2e_ms / 1000.0), "unit": "queries/s",
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "path": "FastPlaid.search(fp32 host queries, top_k) : reload check -> fp16 cast on the host -> "
                        "pinned H2D, search, D2H, sync inside the C-ABI call -> Python list[list[(doc_id, score)]]"},
        "gpu_launches": n_launch * args.steps,
        "clocks": clocks,
        "roofline": {"kernel": ("k5_maxsim_v4_kernel" if Q <= 32 else "k5_maxsim_v5_kernel") +
                               " (fused residual decompression + MaxSim)", "bound": "hbm",
                     "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak if peak else None,
                     "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": ms_bytes, "launch_ms": stage_ms[i_ms]},
        "stages_ms": dict(zip(stage_names, [round(x, 4) for x in stage_ms])),
        "approx_stage": {"mode": args.approx,
                         # two-pass: rows gathered by the bound pass / tokens it walked, and by the exact pass
                         "candidate_tokens_per_step": ap_tokens,
                         "bound_pass_rows_per_token": (k3_stats[0] / k3_stats[1]) if k3_stats[1] else None,
                         "exact_pass_rows_per_token": (k3_stats[2] / k3_stats[1]) if k3_stats[1] else None,
                         "rows_gathered_per_step": (k3_stats[0] + k3_stats[2]) / args.steps,
                         "refined_candidates_per_query_mean": n_refine_mean,
                         "hbm_bytes_per_launch": ap_hbm,
                         "hbm_gbs": ap_hbm / (stage_ms[i_ap] / 1000.0) / 1e9 if stage_ms[i_ap] > 0 else None},
        "wall_s_timed_region": round(t_wall, 3),
    }

    # ---- parity sample (any N) + CPU baseline (N = 1): the oracle on this host's cores ----
    if not args.no_cpu_baseline:
        try:
            # every rank takes part in the engine's side of the check (the sharded search is collective)
            n_par = max(1, min(args.parity_queries, B))
            res_par = fp.search(q_host[0][:n_par], top_k=k, n_full_scores=n_full, n_ivf_probe=N_IVF_PROBE,
                                show_progress=False)
            stg = didx.run_stages(q_dev16[0][:n_par].contiguous(), params, upto="select")
            torch.cuda.synchronize()
            gpu_side = {"S": stg["S"][:, :, :Q].cpu(), "results": res_par}
            if world == 1:
                gpu_side.update(cells=stg["cells"].cpu(), n_cand=stg["n_cand"].cpu(), cand=stg["cand"].cpu(),
                                n_rerank=stg["n_rerank"].cpu(), rerank=stg["rerank"].cpu())
            del stg
            if rank == 0:
                cb, parity = cpu_leg(args, cfg, didx if world == 1 else None, q_host[0], params, gpu_side, world,
                                     device, timed=(world == 1))
                if cb is not None:
                    out["cpu_baseline"] = cb
                out["parity_sample"] = parity
        except Exception as e:  # never lose the GPU numbers
            out["cpu_baseline"] = {"error": repr(e)[:400]}

    # ---- teardown: everything explicit, before the JSON line ----
    del fp
    didx.close()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return out if rank == 0 else {}


def dump_outputs(out_dir: str, ids: torch.Tensor, scores: torch.Tensor, counts: torch.Tensor) -> None:
    """The results of one step as .npy files: ids and counts as float64 (exact for any doc id below 2**53)."""
    os.makedirs(out_dir, exist_ok=True)
    for name, t, dt in (("ids", ids, np.float64), ("scores", scores, np.float32), ("counts", counts, np.float64)):
        np.save(os.path.join(out_dir, f"{name}.npy"), t.cpu().numpy().astype(dt))


def count_launches(world: int, approx: str) -> int:
    """Kernels of OURS per step (memsets/copies not counted): pad, k1, probe, k2 mark+compact, K3 (two-pass: tau,
    hibits, prefix, bound, refine list, prefix, exact; direct: prefix, exact), select, k5, rank; sharded adds the
    key emit, the threshold, the record emit and the merge instead of the rank."""
    k3 = 2 if approx == "direct" else 7
    return 5 + k3 + 1 + 1 + (1 if world == 1 else 4)


# ----------------------------------------------------------------------------------------
# CPU side: the oracle (op-for-op port of the reference's CPU path).  Only this leg and --impl reference use it.
def oracle_index_from_arrays(a):
    from oracle import plaid_oracle as po

    return po.OracleIndex(
        nbits=int(a.nbits),
        centroids=a.centroids.cpu().half(),
        bucket_weights=a.bucket_weights.cpu().half(),
        ivf=a.ivf.cpu().to(torch.int64),
        ivf_lengths=a.ivf_lengths.cpu().to(torch.int64),
        doc_codes=a.doc_codes.cpu().to(torch.int64),
        doc_residuals=a.doc_residuals.cpu(),
        doc_lengths=a.doc_lengths.cpu().to(torch.int64),
    )


def oracle_index_from_device(didx):
    from oracle import plaid_oracle as po

    lens = (didx.doc_offsets[1:] - didx.doc_offsets[:-1]).cpu()
    ivf_len = (didx.ivf_offsets[1:] - didx.ivf_offsets[:-1]).cpu()
    return po.OracleIndex(
        nbits=didx.nbits,
        centroids=didx.centroids.cpu(),
        bucket_weights=didx.bucket_weights.cpu(),
        ivf=didx.ivf_pids.cpu().to(torch.int64) + 0,
        ivf_lengths=ivf_len,
        doc_codes=didx.doc_codes.cpu().to(torch.int64),
        doc_residuals=didx.doc_residuals.cpu(),
        doc_lengths=lens,
    )


def usable_cores() -> int:
    """Host cores this process may actually use (affinity mask and cgroup CPU quota)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()
            if quota != "max":
                n = min(n, max(1, int(float(quota) / float(period) + 0.5)))
    except Exception:
        pass
    return max(1, n)


def pick_threads() -> tuple[int, dict]:
    """ATen's intra-op pool does not scale to every core on a many-core host for this gather-heavy op mix; time a
    representative slice of the approximate stage at a few thread counts and keep the fastest."""
    cores = usable_cores()
    cands = sorted({c for c in (cores, 64, 32, 16, 8) if c <= cores}, reverse=True)
    g = torch.Generator().manual_seed(0)
    S = torch.randn(65536, 32, generator=g).half()
    codes = torch.randint(0, 65536, (600_000,), generator=g)
    mask = torch.ones(2000, 300, 1, dtype=torch.bool)
    timings = {}
    for c in cands:
        torch.set_num_threads(c)
        best = 1e9
        for _ in range(3):
            t0 = time.time()
            x = S.index_select(0, codes).view(2000, 300, 32)
            x = x.masked_fill(mask.expand(2000, 300, 32).logical_not(), -9999.0)
            x.max(dim=1).values.sum(dim=-1, dtype=torch.float32)
            best = min(best, time.time() - t0)
        timings[c] = round(best * 1000, 2)
    pick = min(timings, key=timings.get)
    torch.set_num_threads(pick)
    return pick, timings


def reference_dispatch_workers(num_queries: int) -> int:
    """The reference's CPU dispatch (fast_plaid.py:841-878): more than 10 queries on a CPU-only index are split
    over n_processes = min(num_queries // 10, cpu_count) joblib THREADS, one chunk of queries each."""
    return max(1, min(num_queries // 10, os.cpu_count() or 1))


def time_oracle(po, oidx, queries: torch.Tensor, top_k: int, workers: int) -> float:
    """Seconds for `queries` through the oracle: sequentially (workers = 1) or split over joblib threads the way
    the reference dispatches a CPU batch."""
    def run_chunk(chunk):
        return [po.search_one(q, oidx, N_IVF_PROBE, 2000, N_FULL, top_k, ties="torch") for q in chunk]

    t0 = time.time()
    if workers <= 1:
        run_chunk(queries)
    else:
        from joblib import Parallel, delayed

        size = math.ceil(queries.shape[0] / workers)
        Parallel(n_jobs=workers, prefer="threads")(delayed(run_chunk)(c) for c in torch.split(queries, size))
    return time.time() - t0


def cpu_leg(args, cfg, didx, queries_host: torch.Tensor, params, gpu_side: dict, world: int, device: str,
            timed: bool):
    """Rank 0.  (1) `cpu_baseline` (N = 1 only): the oracle timed on a bounded sample, sequentially and with the
    reference's joblib dispatch.  (2) `parity_sample`: the engine's results for the first queries of the batch
    against the oracle on the FULL index, every difference classified."""
    from oracle import plaid_oracle as po

    cores, thread_timings = pick_threads()
    if didx is not None:
        oidx = oracle_index_from_device(didx)
    else:  # sharded run: rank 0 holds one shard; the oracle needs the whole index (plain torch generator)
        synth = load_synthetic_module()
        full, _ = synth.synthetic_arrays(cfg["n_docs"], cfg["doc_len"], DIM, NBITS, device, SEED_INDEX,
                                         topics=cfg.get("topics", 0), mix=cfg.get("mix", 0.05))
        oidx = oracle_index_from_arrays(full)
        del full
        torch.cuda.empty_cache()
    B = cfg["B"]
    k = params.top_k
    n_par = len(gpu_side["results"])
    keep = PARITY_KEEP

    def pure_run(i):
        st = po.search_one(queries_host[i], oidx, params.n_ivf_probe, 2000, params.n_full_scores, k, ties="canonical",
                           return_stages=True)
        return {key: st[key] for key in keep if key in st}

    # The end-to-end oracle runs of the parity sample double as the CPU baseline (N = 1): the first ones one after the
    # other on one stream, the rest split over joblib threads the way fast_plaid.py:841-878 dispatches a CPU batch.
    from joblib import Parallel, delayed

    workers = reference_dispatch_workers(B)
    cb = None
    if timed and n_par >= 2:
        n_seq = max(1, min(args.cpu_queries or 4, n_par - 1))
        t0 = time.time()
        pure = [pure_run(i) for i in range(n_seq)]
        t_seq = time.time() - t0
        rest = list(range(n_seq, n_par))
        t0 = time.time()
        pure += Parallel(n_jobs=min(workers, len(rest)), prefer="threads")(delayed(pure_run)(i) for i in rest)
        t_disp = time.time() - t0
        v_seq, v_disp = n_seq / t_seq, len(rest) / t_disp
        cb = {"value": max(v_seq, v_disp), "unit": "queries/s", "cores": cores, "kind": "port",
              "sequential_qps": v_seq, "dispatched_qps": v_disp, "dispatch_workers": min(workers, len(rest)),
              "sample": f"sequential: first {n_seq} queries of the batch, one stream, torch intra-op threads={cores} "
                        f"(fastest of {thread_timings} ms on a probe; host has {os.cpu_count()} logical cpus); "
                        f"dispatched: the next {len(rest)} queries over {min(workers, len(rest))} joblib threads, the "
                        f"split fast_plaid.py:841-878 applies to a {B}-query CPU batch; value = the faster of the two; "
                        "full index in both; these runs are also the parity sample's end-to-end oracle runs",
              "seconds": round(t_seq + t_disp, 2)}
    else:
        pure = Parallel(n_jobs=max(1, min(workers, n_par)), prefer="threads")(delayed(pure_run)(i) for i in range(n_par))
    parity = parity_sample(po, oidx, queries_host, params, gpu_side, world, pure)
    return cb, parity


PARITY_KEEP = ("ids", "scores", "cells", "candidates", "approx", "rerank", "exact", "S")


def parity_sample(po, oidx, queries_host, params, gpu, world: int, pure_runs: list | None = None) -> dict:
    """Engine vs oracle on the first queries of a batch, full index, any number of GPUs.

    Two oracle runs per query (canonical tie rule = the engine's):
      pure     : the oracle end to end -- what `identical_id_lists` / `mean_topk_overlap` are measured against;
      given S  : the oracle fed the GPU's own centroid-score table.  The engine's S may differ from ATen's by one
                 fp16 ulp on ~1e-4 of the entries (accumulation order); everything downstream of S is integer work
                 plus the exact scores, so GIVEN S the engine must reproduce the oracle's probed cells, candidates
                 and pruned list exactly, its scores to 1e-3 relative, and its ranking up to ties of those scores.
    Every violation of that chain is an `unexplained_mismatch`.  Differences against the PURE run are then
    classified by where the two oracle runs part: probe boundary (a 1-ulp flip of S moved a probed cell),
    pruning boundary (approximate score at the n_full_scores/4-th), final near-tie (exact score within 1e-3)."""
    from joblib import Parallel, delayed

    results = gpu["results"]
    n = len(results)
    k = params.top_k
    S_gpu = gpu["S"]
    workers = max(1, min(6, n))
    keep = PARITY_KEEP

    def one(i):
        q = queries_host[i]
        if pure_runs is not None:
            pure = pure_runs[i]
        else:
            st = po.search_one(q, oidx, params.n_ivf_probe, 2000, params.n_full_scores, k, ties="canonical",
                               return_stages=True)
            pure = {key: st[key] for key in keep if key in st}
        inj = po.search_one(q, oidx, params.n_ivf_probe, 2000, params.n_full_scores, k, ties="canonical",
                            return_stages=True, inject={"S": S_gpu[i].contiguous()})
        return pure, {key: inj[key] for key in keep if key in inj}

    runs = Parallel(n_jobs=workers, prefer="threads")(delayed(one)(i) for i in range(n))

    identical = identical_given_s = 0
    overlap = 0.0
    unexplained: list[str] = []
    classes = {"probe_boundary": 0, "prune_boundary": 0, "final_near_tie": 0}
    s_ulp_max, s_diff_entries, s_entries = 0, 0, 0
    max_rel = 0.0
    for i, (pure, inj) in enumerate(runs):
        g_ids = [d for d, _ in results[i]]
        g_sc = [s for _, s in results[i]]
        # -- S within one fp16 ulp of ATen's
        if "S" in pure:
            a = S_gpu[i].contiguous().view(torch.int16).to(torch.int32)
            r = pure["S"].contiguous().view(torch.int16).to(torch.int32)
            ka = torch.where(a < 0, -(a & 0x7FFF), a)
            kr = torch.where(r < 0, -(r & 0x7FFF), r)
            dlt = (ka - kr).abs()
            # near zero an fp16 ulp shrinks to 6e-8 while the order-of-summation noise of a 128-term fp32 dot
            # product stays ~1e-5 absolute: entries that differ by more than one ulp must be inside that noise
            far = (dlt > 1) & ((S_gpu[i].float() - pure["S"].float()).abs() > 2e-5)
            s_ulp_max = max(s_ulp_max, int(dlt[(S_gpu[i].float().abs() > 1e-2)].max()) if bool((S_gpu[i].float().abs() > 1e-2).any()) else 0)
            s_diff_entries += int((dlt > 0).sum())
            s_entries += dlt.numel()
            if bool(far.any()):
                unexplained.append(f"q{i}: S differs from the oracle by {int(dlt[far].max())} fp16 ulps / "
                                   f"{float((S_gpu[i].float() - pure['S'].float()).abs().max()):.2e} absolute")
        # -- integer stages given S (one GPU: read from the workspace; sharded: implied by the final result)
        if "cells" in gpu:
            cg = torch.unique(gpu["cells"][i].flatten().long())
            if not torch.equal(cg[cg >= 0], inj["cells"]):
                unexplained.append(f"q{i}: probed cells differ given S")
            nc = int(gpu["n_cand"][i])
            if not torch.equal(gpu["cand"][i, :nc].long(), inj["candidates"]):
                unexplained.append(f"q{i}: candidate ids differ given S")
            nr = int(gpu["n_rerank"][i])
            if not torch.equal(gpu["rerank"][i, :nr].long(), inj["rerank"]):
                # the fp32 summation order of the approximate score differs from ATen's: the pruning boundary may
                # move between candidates whose approximate scores are equal to rounding -- nothing else may
                a_of = dict(zip(inj["candidates"].tolist(), inj["approx"].tolist()))
                ga, ra = set(gpu["rerank"][i, :nr].tolist()), set(inj["rerank"].tolist())
                thr = min(a_of[d] for d in ra) if ra else 0.0
                bad = [d for d in (ga ^ ra) if abs(a_of.get(d, -1e30) - thr) > 1e-6 * max(1.0, abs(thr))]
                if bad:
                    unexplained.append(f"q{i}: pruned list differs given S ({len(bad)} docs off the boundary)")
        # -- final result given S: same documents up to near-ties, scores to 1e-3
        ex_of = dict(zip(inj["rerank"].tolist(), inj["exact"].tolist())) if "rerank" in inj else {}
        for pos, (d, s_) in enumerate(zip(g_ids, g_sc)):
            if d not in ex_of:
                unexplained.append(f"q{i}: returned doc {d} was not in the oracle's pruned list given S")
                continue
            r_ = ex_of[d]
            max_rel = max(max_rel, abs(s_ - r_) / max(1.0, abs(r_)))
            if abs(s_ - r_) > 1e-3 * max(1.0, abs(r_)):
                unexplained.append(f"q{i}: doc {d} score {s_} vs oracle {r_}")
            if pos < len(inj["ids"]) and inj["ids"][pos] != d:
                other = ex_of.get(inj["ids"][pos], None)
                if other is None or abs(other - r_) > 1e-3 * max(1.0, abs(r_)):
                    unexplained.append(f"q{i}: rank {pos}: doc {d} ({r_}) vs oracle doc {inj['ids'][pos]} ({other}): not a near-tie")
        for pos in range(1, len(g_sc)):
            if g_sc[pos] > g_sc[pos - 1]:
                unexplained.append(f"q{i}: returned scores are not sorted at rank {pos}")
        if len(g_ids) != len(inj["ids"]):
            unexplained.append(f"q{i}: {len(g_ids)} results vs {len(inj['ids'])} given S")
        identical_given_s += int(g_ids == inj["ids"])
        # -- against the PURE oracle: headline numbers + classification of every differing document
        identical += int(g_ids == pure["ids"])
        overlap += len(set(g_ids) & set(pure["ids"])) / max(1, len(pure["ids"]))
        if g_ids != pure["ids"]:
            p_cand, i_cand = set(pure["candidates"].tolist()), set(inj["candidates"].tolist())
            p_rr, i_rr = set(pure["rerank"].tolist()), set(inj["rerank"].tolist())
            p_ex = dict(zip(pure["rerank"].tolist(), pure["exact"].tolist()))
            p_kth = pure["scores"][-1] if pure["scores"] else 0.0
            for d in set(g_ids) ^ set(pure["ids"]):
                if (d in p_cand) != (d in i_cand):
                    if torch.equal(pure["cells"], inj["cells"]):
                        unexplained.append(f"q{i}: doc {d} candidate in one run only although the probed cells agree")
                    classes["probe_boundary"] += 1
                elif (d in p_rr) != (d in i_rr):
                    classes["prune_boundary"] += 1
                else:
                    sc = p_ex.get(d, ex_of.get(d))
                    if sc is None or abs(sc - p_kth) > 2e-3 * max(1.0, abs(p_kth)):
                        unexplained.append(f"q{i}: doc {d} (oracle score {sc}) differs from the pure oracle's list "
                                           f"(k-th score {p_kth}) without a boundary to explain it")
                    classes["final_near_tie"] += 1
    return {"queries": n, "n_gpus": world,
            "identical_id_lists": identical, "identical_id_lists_given_gpu_S": identical_given_s,
            "mean_topk_overlap": overlap / max(1, n),
            "S_max_fp16_ulp_above_1e-2": s_ulp_max, "S_entries_differing": s_diff_entries, "S_entries": s_entries,
            "max_rel_score_err_given_S": max_rel,
            "differing_docs_by_cause": classes,
            "unexplained_mismatches": len(unexplained), "unexplained": unexplained[:8],
            "note": "given the GPU's own S the engine must equal the oracle in every integer stage and rank a "
                    "1e-3-valid ordering of its exact scores; differences against the pure oracle are caused by "
                    "1-ulp differences of S (fp32 accumulation order) at a probe / pruning / top-k boundary"}


# ----------------------------------------------------------------------------------------
def run_reference(args) -> dict:
    """The reference's own CPU implementation of the path, i.e. the op-for-op PyTorch-CPU restatement in oracle/
    (the Rust extension cannot be built here: no cargo/rustc), timed on the host cores on the same config and
    synthetic index.  The index and the queries come from plain torch code loaded by file path: this process
    imports neither the engine package nor any of its shared libraries."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return {}
    from oracle import plaid_oracle as po

    cfg = CONFIGS[args.config]
    if not torch.cuda.is_available():  # the GPU only runs the torch ops that GENERATE the synthetic index
        return {"impl": "reference", "unavailable": "no CUDA device to generate the synthetic index"}
    cores, thread_timings = pick_threads()
    synth = load_synthetic_module()
    arrays, _ = synth.synthetic_arrays(cfg["n_docs"], cfg["doc_len"], DIM, NBITS, "cuda:0", SEED_INDEX,
                                       topics=cfg.get("topics", 0), mix=cfg.get("mix", 0.05))
    q_host = make_query_batches(arrays, query_source_docs(cfg["n_docs"]), cfg, N_QUERY_BATCHES)
    oidx = oracle_index_from_arrays(arrays)
    del arrays
    torch.cuda.empty_cache()
    B, k = cfg["B"], cfg["top_k"]
    workers = reference_dispatch_workers(B)
    # one warm-up query, then both dispatch modes once (also warm-up); the faster one is timed
    t0 = time.time()
    po.search_one(q_host[0, 0], oidx, N_IVF_PROBE, 2000, N_FULL, k)
    t_one = time.time() - t0
    n_seq = 2
    v_seq = n_seq / time_oracle(po, oidx, q_host[0, :n_seq], k, 1)
    v_disp = None
    if workers > 1:
        n_d = min(B, workers)
        v_disp = n_d / time_oracle(po, oidx, q_host[1, :n_d], k, workers)
    use_workers = workers if (v_disp or 0.0) > v_seq else 1
    rate = max(v_seq, v_disp or 0.0)
    budget_s = 150.0  # the K timed steps together
    per_step = int(budget_s * rate / max(1, args.steps))
    per_step = max(use_workers, min(B, per_step))
    if use_workers > 1:
        per_step = max(use_workers, per_step // use_workers * use_workers)
    if args.cpu_queries:
        per_step = max(1, min(B, args.cpu_queries))

    t0 = time.time()
    for s in range(args.steps):
        time_oracle(po, oidx, q_host[s % N_QUERY_BATCHES, :per_step], k, use_workers)
    dt = time.time() - t0
    val = per_step * args.steps / dt
    mode = ("split over %d joblib threads like fast_plaid.py:841-878" % use_workers) if use_workers > 1 else "one stream"
    return {
        "impl": "reference",
        "metric": "queries/sec @ top_k=%d, %s-doc/128-dim index; MaxSim HBM GB/s vs roofline" % (
            cfg["top_k"], "1M" if cfg["n_docs"] == 1_000_000 else str(cfg["n_docs"])),
        "value": val, "unit": "queries/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1000.0, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f16", "data": "synthetic (same seeded index and queries as the b200 arm)",
        "config": {"workload": f"{args.config}: {cfg['desc']}", "n_ivf_probe": N_IVF_PROBE, "n_full_scores": N_FULL,
                   "parallelism": "host CPU"},
        "cpu_baseline": {"value": val, "unit": "queries/s", "cores": cores, "kind": "port",
                         "sequential_qps_probe": v_seq, "dispatched_qps_probe": v_disp, "dispatch_workers": workers,
                         "mode_timed": "dispatched" if use_workers > 1 else "sequential",
                         "sample": f"{per_step} queries per step (of the {B}-query batch), full index; {mode} "
                                   f"(the faster of the two modes on a warm-up probe); torch intra-op threads={cores} "
                                   f"(fastest of {thread_timings} ms on a probe; host has {os.cpu_count()} logical "
                                   f"cpus); first query took {t_one:.1f} s"},
        "e2e": {"value": val, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed steps (at least 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--config", choices=list(CONFIGS), default="cfg3")
    ap.add_argument("--cpu-queries", type=int, default=0, help="queries timed on the CPU (0 = auto)")
    ap.add_argument("--parity-queries", type=int, default=PARITY_QUERIES,
                    help="queries cross-checked against the oracle (rank 0, any number of GPUs)")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the oracle legs (CPU baseline and parity sample)")
    ap.add_argument("--query-groups", type=int, default=0,
                    help="multi-GPU runs: query groups of the rank grid (0 = as many as the index size allows: fewest document "
                         "shards that fit the per-GPU budget)")
    ap.add_argument("--approx", choices=["two-pass", "direct"], default="two-pass",
                    help="approximate stage: exact two-pass pruning (default) or the one-pass A/B alternative")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the ids, scores and counts the timed path returned in its last step to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the engine's results: it needs --impl b200")
    # keep stdout clean for the ONE JSON line: NCCL / libraries may print to fd 1
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    out = run_reference(args) if args.impl == "reference" else run_b200(args)
    sys.stdout.flush()
    if out:
        os.write(real_stdout, (json.dumps(out) + "\n").encode())


if __name__ == "__main__":
    main()
