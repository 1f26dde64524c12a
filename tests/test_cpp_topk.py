"""Top-k sampling through the C++ host layer (tests/cpp/host_topk_test.cc): Options::top_k on Blocking and Async,
Async pooling only equal top_k, the std::invalid_argument cases, the pivot and one text-level request.  GPU: its answers
equal the C ABI's slimt_b200_translate_topk with each segment's FNV-1a key.  (That the program builds is checked on the
CPU by test_capi_topk.py.)"""
import os
import struct
import subprocess

import numpy as np
import pytest

from slimt_b200 import synth
from test_cpp_sampling import fnv1a64

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "tests", "cpp", "host_topk_test")
SPM = os.path.join(ROOT, "tests", "golden", "text", "spm_unigram.model")


def _build():
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "slimt_b200", "csrc"), "host_topk"])
    assert os.path.exists(BIN)


@pytest.mark.gpu
def test_service_topk_matches_ctypes(gpu_ctx, tiny_model, shortlist_assets, tmp_path):
    from slimt_b200 import capi
    _build()
    path, _ = tiny_model
    sl_path, _ = shortlist_assets
    sents = synth.make_sentences(20, (2, 12), seed=93)
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
    assert "host_topk_test ok" in r.stdout
    assert int(next(l for l in r.stdout.split("\n") if l.startswith("text sentences ")).split()[2]) >= 1
    buf = open(tmp_path / "o.bin", "rb").read()
    m = capi.Model(gpu_ctx, open(path, "rb").read())
    keys = np.array([fnv1a64(s) for s in sents], dtype=np.uint64)
    outs, st = m.translate(sents, max_words=96, shortlist_bin=open(sl_path, "rb").read(), want_scores=True,
                           sampling={"temperature": 0.8, "seed": 7, "keys": keys, "top_k": 10})
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
