"""bench.py's workload table: every BASELINE.json GPU config has an entry, the headline is the default, and the
synthetic inputs each entry describes can be built and batched on the CPU (no GPU work)."""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from slimt_b200 import capi, synth  # noqa: E402


def test_every_baseline_gpu_config_has_a_workload():
    baseline = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert len(baseline["configs"]) == 5
    # configs[0] CPU-runnable case, [1] headline, [2] base, [3] no shortlist, [4] mixed lengths
    assert {"tiny_b64", "tiny_shortlist", "base_shortlist", "tiny_full", "mixed"} <= set(bench.WORKLOADS)
    assert bench.WL is bench.WORKLOADS["tiny_shortlist"]
    head = bench.WORKLOADS["tiny_shortlist"]
    assert head["sentences"] == 4096 and head["length"] == 32 and head["shortlist"] and head["dims"] == "TINY"
    assert not bench.WORKLOADS["tiny_full"]["shortlist"]
    assert getattr(synth, bench.WORKLOADS["base_shortlist"]["dims"]).emb == 512
    assert bench.WORKLOADS["mixed"]["length"] == (8, 256)


def test_mixed_workload_batches_respect_max_words():
    wl = bench.WORKLOADS["mixed"]
    sents = synth.make_sentences(2048, wl["length"], seed=5)
    lens = [len(s) for s in sents]
    assert min(lens) >= 8 and max(lens) <= 256 and all(s[-1] == 0 for s in sents)
    plan = capi.batcher_plan(lens, wl["max_words"])
    seen = sorted(i for ids, _ in plan for i in ids)
    assert seen == list(range(len(sents)))
    for ids, width in plan:
        assert width == max(lens[i] for i in ids)
        assert len(ids) * width <= wl["max_words"]
    # ascending-length greedy batching (Batcher.cc:95-120): widths never decrease
    widths = [w for _, w in plan]
    assert widths == sorted(widths)


def test_dump_outputs_whole_below_the_cap_and_a_fixed_sample_above(tmp_path, monkeypatch):
    arrays = {"exact_step_tokens_000": np.arange(3000, dtype=np.float32).reshape(60, 50),
              "exact_e2e_offsets": np.arange(1001, dtype=np.float64)}
    bench.dump_outputs(str(tmp_path / "whole"), arrays)
    for name, a in arrays.items():
        got = np.load(tmp_path / "whole" / f"{name}.npy")
        assert got.dtype == a.dtype and np.array_equal(got, a)
    monkeypatch.setattr(bench, "DUMP_CAP_BYTES", 4096)
    bench.dump_outputs(str(tmp_path / "a"), arrays)
    bench.dump_outputs(str(tmp_path / "b"), arrays)
    total = 0
    for name, a in arrays.items():
        x, y = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert x.dtype == a.dtype and np.array_equal(x, y) and 0 < x.size < a.size
        assert np.all(np.diff(x) > 0)  # elements of the original, in their original order
        total += x.nbytes
    assert total <= 4096


def test_headline_is_one_batch_of_4096_by_32():
    wl = bench.WORKLOADS["tiny_shortlist"]
    plan = capi.batcher_plan([wl["length"]] * wl["sentences"], wl["max_words"])
    assert len(plan) == 1 and len(plan[0][0]) == 4096 and plan[0][1] == 32
    assert np.float32(bench.LIMIT) * np.float32(32) == 48.0
