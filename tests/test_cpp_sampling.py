"""Sampling through the C++ host layer (tests/cpp/host_sampling_test.cc): Options::sample on Blocking and Async,
pooled Async requests, the cache bypass, the pivot and one text-level request.  CPU: the program builds.  GPU: its
answers equal the C ABI's slimt_b200_translate_sampled with each segment's FNV-1a key."""
import os
import struct
import subprocess

import numpy as np
import pytest

from slimt_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "tests", "cpp", "host_sampling_test")
SPM = os.path.join(ROOT, "tests", "golden", "text", "spm_unigram.model")


def _build():
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "slimt_b200", "csrc"), "host_sampling"])
    assert os.path.exists(BIN)


def fnv1a64(words):
    """The services' sampling key: 64-bit FNV-1a over the words' little-endian bytes."""
    h = 0xcbf29ce484222325
    for b in np.asarray(words, dtype="<u4").tobytes():
        h = ((h ^ b) * 0x100000001b3) & 0xFFFFFFFFFFFFFFFF
    return h


def test_sampling_program_builds():
    _build()


def test_fnv1a64_known_answers():
    # FNV-1a 64 of the empty input is the offset basis; of the bytes 61 00 00 00 ("a" as one little-endian u32)
    assert fnv1a64([]) == 0xcbf29ce484222325
    h = 0xcbf29ce484222325
    for b in b"a\0\0\0":
        h = ((h ^ b) * 0x100000001b3) & 0xFFFFFFFFFFFFFFFF
    assert fnv1a64([ord("a")]) == h


@pytest.mark.gpu
def test_service_sampling_matches_ctypes(gpu_ctx, tiny_model, shortlist_assets, tmp_path):
    from slimt_b200 import capi
    _build()
    path, _ = tiny_model
    sl_path, _ = shortlist_assets
    sents = synth.make_sentences(20, (2, 12), seed=92)
    with open(tmp_path / "s.u32", "wb") as f:
        f.write(struct.pack("<I", len(sents)))
        for s in sents:
            f.write(struct.pack("<I", len(s)) + np.asarray(s, dtype=np.uint32).tobytes())
    text_model = str(tmp_path / "text.bin")
    synth.write_model(text_model, synth.make_params(synth.ModelDims(vocab=1024), seed=77, eos_bias=3.0))
    text = "Hello world. This is a second sentence, with a comma."
    r = subprocess.run([BIN, path, sl_path, str(tmp_path / "s.u32"), str(tmp_path / "o.bin"), text_model, SPM, text],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "host_sampling_test ok" in r.stdout
    assert int(next(l for l in r.stdout.split("\n") if l.startswith("text sentences ")).split()[2]) >= 1
    buf = open(tmp_path / "o.bin", "rb").read()
    m = capi.Model(gpu_ctx, open(path, "rb").read())
    keys = np.array([fnv1a64(s) for s in sents], dtype=np.uint64)
    outs, st = m.translate(sents, max_words=96, shortlist_bin=open(sl_path, "rb").read(), want_scores=True,
                           sampling={"temperature": 0.8, "seed": 7, "keys": keys})
    n, = struct.unpack_from("<I", buf, 0)
    pos = 4
    assert n == len(sents)
    for i in range(n):
        ln, = struct.unpack_from("<I", buf, pos)
        pos += 4
        words = np.frombuffer(buf, dtype=np.uint32, count=ln, offset=pos)
        pos += 4 * ln
        scores = np.frombuffer(buf, dtype=np.float32, count=ln, offset=pos)
        pos += 4 * ln
        assert words.tolist() == outs[i].tolist()
        assert np.array_equal(scores, st["scores"][i])
    m.close()
