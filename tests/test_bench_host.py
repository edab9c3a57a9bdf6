"""CPU checks of bench.py's host-side pieces: the synthetic workload generator (planted pages, topic model), the JSON keys
of the reference arm, and the flag defaults the driver relies on (no GPU, no oracle compute beyond a tiny sample)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402


def test_synthetic_shard_is_unit_norm_with_planted_and_topic_structure(monkeypatch):
    monkeypatch.setattr(bench, "N_TOPICS", 8)
    dev = torch.device("cpu")
    anchors = bench.topic_anchors(dev)
    q = bench.make_queries(2)
    assert torch.equal(q, bench.make_queries(2)) and q.shape == (64, 128)  # identical on every rank
    packed, planted = bench.build_shard(64, dev, 1, q, planted_per_query=2, topic_pages=32, anchors=anchors)
    assert packed.data_ptr() % 1024 == 0 and packed.numel() == 64 * 1024 * 256
    rows = packed.view(torch.bfloat16).view(-1, 128).float()
    assert torch.isfinite(rows).all() and abs(float(rows.norm(dim=1).mean()) - 1.0) < 1e-2
    assert all(p >= 32 for ids in planted.values() for p in ids)  # planted pages never overwrite topic pages

    def maxsim(qq):
        return (qq @ rows.T).view(qq.shape[0], 64, 1024).max(dim=2)[0].sum(0)

    for qi in range(2):  # a planted page is the exhaustive top-1 of its query
        assert int(maxsim(q[qi * 32:(qi + 1) * 32]).argmax()) in planted[qi]
    tq, topics = bench.make_topic_queries(3, anchors)
    s = maxsim(tq[:32])
    same = [p for p in range(32) if p % 8 == topics[0]]
    other = [p for p in range(32) if p % 8 != topics[0]]
    assert s[same].mean() > s[other].mean() + 3.0  # topic pages answer topic queries ...
    assert s[same].max() - s[same].min() > 0.5      # ... to different degrees (coverage x noise): graded relevance


def test_reference_arm_line_has_the_contract_keys():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--ref-budget", "0.5"], capture_output=True, text=True, timeout=300, check=True).stdout.strip().splitlines()
    line = json.loads(out[-1])
    assert line["impl"] == "reference" and line["metric"] == bench.METRIC and line["unit"] == bench.UNIT
    assert line["higher_is_better"] is True and line["cpu_baseline"]["kind"] == "port" and line["gpu_launches"] == 0
    assert line["e2e"] == {"value": line["value"], "unit": bench.UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_defaults_finish_within_minutes():
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert 'ap.add_argument("--gpus", type=int, default=1)' in src
    assert 'ap.add_argument("--pages", type=int, default=524288' in src  # the largest resident shard (SURVEY 8d)
    assert np.prod([524288, 1024, 256]) < 180e9


def test_dump_outputs_writes_float_arrays_and_enforces_the_size_limit(tmp_path):
    ids = np.array([[3, 2 ** 40 + 1]], dtype=np.int64)
    scores = np.array([[1.5, -0.25]], dtype=np.float32)
    bench.dump_outputs(str(tmp_path / "out"), {"topk_scores": scores, "topk_ids": ids})
    got_s, got_i = np.load(tmp_path / "out" / "topk_scores.npy"), np.load(tmp_path / "out" / "topk_ids.npy")
    assert got_s.dtype == np.float32 and np.array_equal(got_s, scores)
    assert got_i.dtype == np.float64 and np.array_equal(got_i.astype(np.int64), ids)
    with pytest.raises(ValueError):
        bench.dump_outputs(str(tmp_path / "big"), {"x": np.zeros((1 << 20) + 1, dtype=np.float64)}, limit_bytes=8 << 20)
    assert not (tmp_path / "big").exists()
