"""Beam search through the C++ host layer (tests/cpp/host_beam_test.cc): Options::beam_size on Blocking, the cache
bypass, and sample with a beam refused.  CPU: the program builds.  GPU: beam_size 4 returns slimt_b200_translate_beam's
best words, scores and alignments, and beam_size 1 returns what the greedy call returns."""
import os
import struct
import subprocess

import numpy as np
import pytest

from slimt_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "tests", "cpp", "host_beam_test")


def _build():
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "slimt_b200", "csrc"), "host_beam"])
    assert os.path.exists(BIN)


def test_beam_program_builds():
    _build()


def _read(buf, pos):
    n, = struct.unpack_from("<I", buf, pos)
    pos += 4
    out = []
    for _ in range(n):
        ln, src = struct.unpack_from("<II", buf, pos)
        pos += 8
        words = np.frombuffer(buf, dtype=np.uint32, count=ln, offset=pos)
        pos += 4 * ln
        scores = np.frombuffer(buf, dtype=np.float32, count=ln, offset=pos)
        pos += 4 * ln
        align = np.frombuffer(buf, dtype=np.float32, count=ln * src, offset=pos).reshape(ln, src)
        pos += 4 * ln * src
        out.append((words, scores, align))
    return out, pos


@pytest.mark.gpu
def test_service_beam_matches_ctypes(gpu_ctx, tiny_model, shortlist_assets, tmp_path):
    from slimt_b200 import capi
    _build()
    path, _ = tiny_model
    sl_path, _ = shortlist_assets
    sents = synth.make_sentences(20, (2, 12), seed=93)
    with open(tmp_path / "s.u32", "wb") as f:
        f.write(struct.pack("<I", len(sents)))
        for s in sents:
            f.write(struct.pack("<I", len(s)) + np.asarray(s, dtype=np.uint32).tobytes())
    r = subprocess.run([BIN, path, sl_path, str(tmp_path / "s.u32"), str(tmp_path / "o.bin")], capture_output=True,
                       text=True)
    assert r.returncode == 0, r.stderr
    assert "host_beam_test ok" in r.stdout
    buf = open(tmp_path / "o.bin", "rb").read()
    b4, pos = _read(buf, 0)
    b1, pos = _read(buf, pos)
    assert pos == len(buf)
    m = capi.Model(gpu_ctx, open(path, "rb").read())
    try:
        sl = open(sl_path, "rb").read()
        _, st = m.translate_beam(sents, 96, 4, 1, 1.0, shortlist_bin=sl, want_alignments=True)
        outs, gst = m.translate(sents, max_words=96, shortlist_bin=sl, want_scores=True, want_alignments=True)
    finally:
        m.close()
    for i in range(len(sents)):
        assert b4[i][0].tolist() == st["tokens"][i].tolist()
        assert np.array_equal(b4[i][1].view(np.uint32), st["scores"][i].view(np.uint32))
        assert np.array_equal(b4[i][2].view(np.uint32), st["alignments"][i].view(np.uint32))
        assert b1[i][0].tolist() == outs[i].tolist()
        assert np.array_equal(b1[i][1].view(np.uint32), gst["scores"][i].view(np.uint32))
        assert np.array_equal(b1[i][2].view(np.uint32), gst["alignments"][i].view(np.uint32))
