"""Scoring through the C++ host layer (tests/cpp/host_score_test.cc): Blocking::score with alignments, its refusal of
Options::sample and its bypass of the translation cache.  CPU: the program builds.  GPU: its scores and alignments
equal the C ABI's slimt_b200_score, bit for bit."""
import os
import struct
import subprocess

import numpy as np
import pytest

from slimt_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "tests", "cpp", "host_score_test")


def _build():
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "slimt_b200", "csrc"), "host_score"])
    assert os.path.exists(BIN)


def test_score_program_builds():
    _build()


@pytest.mark.gpu
def test_blocking_score_matches_ctypes(gpu_ctx, tiny_model, shortlist_assets, tmp_path):
    from slimt_b200 import capi
    _build()
    path, _ = tiny_model
    sl_path, _ = shortlist_assets
    sources = synth.make_sentences(20, (2, 12), seed=93)
    rng = np.random.default_rng(94)
    targets = [rng.integers(0, 32000, size=int(rng.integers(0, 20))).astype(np.uint32) for _ in sources]
    with open(tmp_path / "p.u32", "wb") as f:
        f.write(struct.pack("<I", len(sources)))
        for s, t in zip(sources, targets):
            f.write(struct.pack("<I", len(s)) + np.asarray(s, dtype=np.uint32).tobytes())
            f.write(struct.pack("<I", len(t)) + t.tobytes())
    r = subprocess.run([BIN, path, sl_path, str(tmp_path / "p.u32"), str(tmp_path / "o.bin")], capture_output=True,
                       text=True)
    assert r.returncode == 0, r.stderr
    m = capi.Model(gpu_ctx, open(path, "rb").read())
    try:
        want, st = m.score(sources, targets, max_words=96, shortlist_bin=open(sl_path, "rb").read(),
                           want_alignments=True)
    finally:
        m.close()
    raw = np.fromfile(tmp_path / "o.bin", dtype=np.uint32)
    pos = 0
    for i, (s, t) in enumerate(zip(sources, targets)):
        n = int(raw[pos])
        pos += 1
        assert n == len(t)
        assert np.array_equal(raw[pos:pos + n], want[i].view(np.uint32)), f"scores of pair {i}"
        pos += n
        assert np.array_equal(raw[pos:pos + n * len(s)], st["alignments"][i].reshape(-1).view(np.uint32)), f"alignment {i}"
        pos += n * len(s)
    assert pos == len(raw)
