"""GPU: the output GEMM's bound-filter encoding (out_argmax.cu).  By default the fused argmax adds every column's
offset round(bias * aq * bq) on the tensor core as 32 int8 digits, which hold at most 500 093 in magnitude.  A model
with an output bias beyond that range decodes through the bound filter instead, with the full vocabulary and with a
shortlist, in both arithmetic modes."""
import struct

import numpy as np
import pytest

import sb_testutil as util
from oracle import slimt_oracle as so
from slimt_b200 import capi, synth

pytestmark = pytest.mark.gpu
DIGIT_RANGE = 500093  # largest |offset| the digits represent (out_argmax.cu, out_ext_kernel)
BIASED_COLUMN = 5     # not EOS (synth.EOS_ID)


def _write_fallback_model(tmp_path_factory, cfg, name):
    """The synthetic model `cfg` with one output column biased so far below the others that it never wins, and whose
    offset is four times what the digits hold."""
    items = synth.make_params(cfg, seed=1234)
    typ, shape, blob = items["Wemb"]
    V, E = shape
    bq = struct.unpack("<f", blob[V * E:V * E + 4])[0]
    aq = float(np.frombuffer(items["none_QuantMultA"][2], dtype=np.float32)[0])
    typ, shape, blob = items["decoder_ff_logit_out_b"]
    b = np.frombuffer(blob, dtype=np.float32).copy()
    b[BIASED_COLUMN] = np.float32(-4.0 * DIGIT_RANGE / (aq * bq))
    items["decoder_ff_logit_out_b"] = (typ, shape, b.tobytes())
    offset = abs(float(b[BIASED_COLUMN]) * aq * bq)
    # past the digits (so the bound filter runs), inside the bound filter's exact-integer range
    assert 2 * DIGIT_RANGE < offset < 2 ** 23, offset
    assert BIASED_COLUMN != synth.EOS_ID
    path = str(tmp_path_factory.mktemp("model") / f"{name}_out_fallback.bin")
    synth.write_model(path, items)
    return path, synth.read_model(path)


@pytest.fixture(scope="module")
def fallback_model(tmp_path_factory):
    """tiny11 (E = 256: the bound filter at K = 256) with the biased column."""
    return _write_fallback_model(tmp_path_factory, synth.TINY, "tiny11")


@pytest.fixture(scope="module")
def fallback_base_model(tmp_path_factory):
    """The base model (E = 512: the bound filter at K = 512) with the same biased column."""
    return _write_fallback_model(tmp_path_factory, synth.BASE, "base")


def test_exact_greedy_tokens_equal_oracle(gpu_ctx, fallback_model):
    path, items = fallback_model
    m = capi.Model(gpu_ctx, open(path, "rb").read())
    orc = so.Oracle(items)
    sents = synth.make_sentences(40, (2, 30), seed=11)
    tokens, lengths = util.pad_batch(sents)
    ref = orc.forward(tokens, lengths)
    assert not (np.asarray(ref["step_tokens"]) == BIASED_COLUMN).any()
    out = m.forward(tokens, lengths)
    assert out["steps"] == len(ref["step_tokens"])
    assert np.array_equal(out["step_tokens"], ref["step_tokens"])
    fr, offs, lists = synth.make_shortlist(vocab=32000, frequent=100, best=100, seed=7)
    sl = so.shortlist_generate(np.concatenate(sents), fr, offs, lists, 32000)
    ref_sl = orc.forward(tokens, lengths, shortlist=sl)
    out_sl = m.forward(tokens, lengths, shortlist=sl)
    assert out_sl["steps"] == len(ref_sl["step_tokens"])
    assert np.array_equal(out_sl["step_tokens"], ref_sl["step_tokens"])
    m.close()


def test_tolerance_mode_fused_argmax_agrees_with_logits(fallback_model):
    """Teacher forcing keeps the histories equal; the fused argmax (the bound filter's exact first maximum of the
    accumulators, in tolerance mode too) must agree with the argmax of the same mode's float logits except at
    near-ties (the bar of test_teacher_forced_logits_within_rtol)."""
    path, _ = fallback_model
    ctx = capi.Context(0)
    ctx.set_math(True)
    m = capi.Model(ctx, open(path, "rb").read())
    sents = synth.make_sentences(24, (3, 30), seed=5)
    tokens, lengths = util.pad_batch(sents)
    steps = int(np.float32(1.5) * np.float32(tokens.shape[1]))
    forced = np.random.RandomState(3).randint(1, 32000, size=(steps, len(sents))).astype(np.uint32)
    tap = m.forward(tokens, lengths, forced=forced, want_logits=True)
    fused = m.forward(tokens, lengths, forced=forced)
    agree = (fused["step_tokens"] == tap["step_tokens"]).mean()
    assert agree >= 0.999, agree
    m.close()
    ctx.close()
