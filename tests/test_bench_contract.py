"""bench.py contract pieces that can be checked without a GPU: the reference arm answers with one
JSON line (never a traceback) and the product arm refuses to run without CUDA instead of falling
back to a CPU path."""

from __future__ import annotations

import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
no_gpu = pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")


@no_gpu
def test_reference_arm_prints_one_json_line_without_a_gpu():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-500:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and "unavailable" in d


@no_gpu
def test_product_arm_has_no_cpu_fallback():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode != 0
    assert "CUDA" in (r.stderr + r.stdout)


def test_steps_below_one_are_refused():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 2 and "--steps" in r.stderr


def test_dump_outputs_writes_float_arrays_of_the_results(tmp_path):
    sys.path.insert(0, ROOT)
    import bench

    ids = torch.tensor([[7, 2**40 + 3, -1], [0, -1, -1]])
    scores = torch.tensor([[31.5, 30.25, float("-inf")], [12.0, float("-inf"), float("-inf")]])
    counts = torch.tensor([2, 1], dtype=torch.int32)
    out = tmp_path / "dump"
    bench.dump_outputs(str(out), ids, scores, counts)
    got = {p.stem: np.load(p) for p in out.iterdir()}
    assert set(got) == {"ids", "scores", "counts"}
    assert got["ids"].dtype == np.float64 and got["ids"].tolist() == ids.tolist()
    assert got["scores"].dtype == np.float32 and got["scores"].tolist() == scores.tolist()
    assert got["counts"].dtype == np.float64 and got["counts"].tolist() == counts.tolist()


def test_bench_configs_cover_the_baseline_configs():
    sys.path.insert(0, ROOT)
    import bench

    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert {"cfg2", "cfg3", "cfg4", "cfg5"} <= set(bench.CONFIGS)
    assert bench.CONFIGS["cfg3"]["n_docs"] == 1_000_000 and bench.CONFIGS["cfg3"]["top_k"] == 100
    assert "north_star" in base


def test_grid_policy_uses_the_fewest_document_shards_that_fit():
    """bench.default_query_groups: every rank a query group while the index fits one GPU's budget, document shards
    (always a divisor of the world size) only when it does not."""
    sys.path.insert(0, ROOT)
    import bench
    from fast_plaid_b200.engine import shard_grid

    for world in (1, 2, 4, 8):
        assert bench.default_query_groups(world, bench.CONFIGS["cfg3"]) == world
    big = dict(n_docs=10_000_000, doc_len=300)  # ~220 GB of index data
    assert bench.default_query_groups(8, big) == 2  # 4 shards of 55 GB, two query groups
    assert bench.default_query_groups(4, big) == 1
    assert bench.default_query_groups(2, big) == 1  # does not fit at all: as many shards as there are ranks
    for world in (2, 4, 8):
        g = bench.default_query_groups(world, big)
        cells = {shard_grid(r, world, g)[:2] for r in range(world)}
        assert len(cells) == world and world % g == 0


def test_parity_sample_classifier_on_an_oracle_stand_in():
    """bench.parity_sample, fed the oracle's own results in place of the engine's: nothing to explain, every list
    identical; and with one returned document swapped for a far-away one it must report the mismatch."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import bench
    from util import build_oracle_index, make_docs, make_queries

    from oracle import plaid_oracle as po

    docs = make_docs(300, 10, 40, seed=3)
    oidx, _ = build_oracle_index(docs, kmeans_niters=2)
    queries = make_queries(4, 16, seed=5, docs=docs)

    class P:
        n_ivf_probe, n_full_scores, top_k = 4, 64, 5

    S, results, stages = [], [], []
    for b in range(4):
        st = po.search_one(queries[b], oidx, 4, 2000, 64, 5, ties="canonical", return_stages=True)
        S.append(st["S"])
        results.append(list(zip(st["ids"], st["scores"])))
        stages.append(st)
    gpu = {"S": torch.stack(S), "results": results}
    out = bench.parity_sample(po, oidx, queries, P, gpu, world=2)
    assert out["queries"] == 4 and out["identical_id_lists"] == 4 and out["identical_id_lists_given_gpu_S"] == 4
    assert out["unexplained_mismatches"] == 0 and out["S_max_fp16_ulp_above_1e-2"] == 0
    # single-GPU form: the integer stages are compared too
    R = max(len(s["rerank"]) for s in stages)
    C = max(len(s["candidates"]) for s in stages)
    cells = torch.full((4, 16, 4), -1, dtype=torch.int32)
    cand = torch.zeros((4, C), dtype=torch.int32)
    rer = torch.zeros((4, R), dtype=torch.int32)
    for b, s in enumerate(stages):
        cells[b].view(-1)[: s["probe_cells"].numel()] = s["probe_cells"].to(torch.int32)
        cand[b, : len(s["candidates"])] = s["candidates"].to(torch.int32)
        rer[b, : len(s["rerank"])] = s["rerank"].to(torch.int32)
    gpu1 = dict(gpu, cells=cells, cand=cand, rerank=rer,
                n_cand=torch.tensor([len(s["candidates"]) for s in stages]),
                n_rerank=torch.tensor([len(s["rerank"]) for s in stages]))
    assert bench.parity_sample(po, oidx, queries, P, gpu1, world=1)["unexplained_mismatches"] == 0
    # a wrong document in the result must not pass
    bad = [list(r) for r in results]
    worst = int(stages[0]["rerank"][stages[0]["exact"].argmin()])
    if worst != bad[0][0][0]:
        bad[0][0] = (worst, bad[0][0][1])
        out = bench.parity_sample(po, oidx, queries, P, dict(gpu, results=bad), world=2)
        assert out["unexplained_mismatches"] > 0
