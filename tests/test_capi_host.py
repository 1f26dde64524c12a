"""CPU: the C-ABI library loads without a GPU, exports every symbol include/*.h declares, and its host-side
logic (Batcher, ShortlistGenerator, weight prepare) matches the reference semantics.  No compute calls."""
import ctypes
import os
import re

import numpy as np
import pytest

import sb_testutil as util
from oracle import slimt_oracle as so
from slimt_b200 import capi, synth


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(util.ROOT, "include", "slimt_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(slimt_b200_[a-z0-9_]+)\s*\(", header)))
    assert len(declared) >= 20
    lib = ctypes.CDLL(capi.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/slimt_b200.h but not exported"
    assert sorted(capi.EXPORTS) == declared


def test_context_creation_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(RuntimeError, match="no CUDA device|CUDA"):
        capi.Context(0)


@pytest.mark.parametrize("max_words", [18, 64, 1024, 5])
def test_batcher_plan_matches_reference_policy(max_words):
    rng = np.random.RandomState(max_words)
    lengths = rng.randint(1, 17, size=200)
    got = capi.batcher_plan(lengths, max_words)
    want = util.batcher_generate_py(lengths, max_words)
    assert [(ids.tolist(), w) for ids, w in got] == want
    seen = np.concatenate([ids for ids, _ in got])
    assert sorted(seen.tolist()) == list(range(200))
    for ids, w in got:
        assert w == max(lengths[i] for i in ids)
        assert len(ids) * w <= max_words or len(ids) == 1


def test_batcher_plan_empty_and_single():
    assert capi.batcher_plan([], 100) == []
    got = capi.batcher_plan([7], 100)
    assert len(got) == 1 and got[0][0].tolist() == [0] and got[0][1] == 7


def test_shortlist_generate_matches_oracle(shortlist_assets):
    path, (fr, offs, lists) = shortlist_assets
    blob = open(path, "rb").read()
    rng = np.random.RandomState(0)
    for n in (1, 7, 300):
        words = rng.randint(0, 32000, size=n).astype(np.uint32)
        a = capi.shortlist_generate(blob, words, 32000)
        b = so.shortlist_generate(words, fr, offs, lists, 32000)
        assert np.array_equal(a, b) and len(a) % 8 == 0


def test_shortlist_rejects_bad_images(tmp_path):
    with pytest.raises(RuntimeError, match="too short"):
        capi.shortlist_generate(b"\0" * 8, np.zeros(1, np.uint32), 10)
    fr, offs, lists = synth.make_shortlist(vocab=100, frequent=5, best=3, seed=1, spread=10)
    p = str(tmp_path / "sl_bad.bin")
    synth.write_shortlist(p, fr, offs, lists, best=3)
    blob = bytearray(open(p, "rb").read())
    with pytest.raises(RuntimeError, match="file size"):
        capi.shortlist_generate(bytes(blob[:-4]), np.zeros(1, np.uint32), 100)
    blob[0] ^= 0xFF
    with pytest.raises(RuntimeError, match="magic"):
        capi.shortlist_generate(bytes(blob), np.zeros(1, np.uint32), 100)


def test_shortlist_check_and_corrupt_contents(tmp_path):
    """check = true of the reference's loader (Shortlist.cc:16-37, 68-98): checksum + content_check.  With or without
    it, an image whose offsets or ids point outside their tables is reported, never followed."""
    import struct
    fr, offs, lists = synth.make_shortlist(vocab=100, frequent=5, best=3, seed=1, spread=10)
    p = str(tmp_path / "sl_chk.bin")
    synth.write_shortlist(p, fr, offs, lists, best=3, checksum=True)
    good = open(p, "rb").read()
    capi.shortlist_check(good, 100)
    words = np.array([1, 2, 3, 50], dtype=np.uint32)
    assert len(capi.shortlist_generate(good, words, 100)) % 8 == 0
    flipped = bytearray(good)
    flipped[-1] ^= 0x01  # a target id changes: the checksum no longer matches
    with pytest.raises(RuntimeError, match="checksum"):
        capi.shortlist_check(bytes(flipped), 100)
    with pytest.raises(RuntimeError, match="out of bounds"):
        capi.shortlist_check(good, 50)  # image built for a larger vocabulary than the model's
    with pytest.raises(RuntimeError, match="out of bounds"):
        capi.shortlist_generate(good, words, 50)
    # an offset beyond the list table
    bad = bytearray(good)
    struct.pack_into("<Q", bad, 48 + 8 * 3, 1 << 40)
    with pytest.raises(RuntimeError, match="offset table"):
        capi.shortlist_generate(bytes(bad), words, 100)
    # a header whose counts would overflow the size arithmetic
    huge = bytearray(good)
    struct.pack_into("<QQ", huge, 32, (1 << 61) + 3, 1 << 62)
    with pytest.raises(RuntimeError, match="file size"):
        capi.shortlist_generate(bytes(huge), words, 100)
    # source word id 0xFFFFFFFF must not wrap the `word + 1` bound
    assert len(capi.shortlist_generate(good, np.array([0xFFFFFFFF, 3], dtype=np.uint32), 100)) % 8 == 0


def test_prepare_weight_entry_points():
    lib = capi.lib()
    rng = np.random.RandomState(2)
    Bt = rng.randint(-127, 128, size=(64, 128)).astype(np.int8)
    out = np.zeros_like(Bt)
    lib.slimt_b200_qmm_prepare_weight_quantized_transposed(Bt.ctypes.data, out.ctypes.data, 128, 64)
    assert np.array_equal(out, Bt)  # logical layout [N][K] preserved: compare in logical order (appendix A.2)
    w = (rng.standard_normal((64, 128)) * 0.2).astype(np.float32)
    w[0, :4] = [1e9, -1e9, 0.5 / 300, -128.0 / 300]
    q = np.zeros((64, 128), dtype=np.int8)
    lib.slimt_b200_qmm_prepare_weight_transposed(w.ctypes.data, q.ctypes.data, ctypes.c_float(300.0), 128, 64)
    assert np.array_equal(q, so.quantize(w, 300.0)) and q.min() >= -127
