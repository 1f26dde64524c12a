"""GPU: slimt_b200_score at the batch level, where the scoring pass differs from the step path.

Padded target positions: a sentence's scores and alignments do not depend on the longer targets it shares a batch
with.  Output row chunks: the output stage scores the M = B * T_target rows in chunks of 16 k rows, each with its own
offsets into the targets, the scores and the output operand; batches of more than one chunk, with a last chunk that is
not a multiple of 128 rows and at the headline shape, are compared with the step path bit for bit at every position."""
import numpy as np
import pytest

from slimt_b200 import capi, synth
from test_gpu_score import BIG, NO_EOS_BIAS, _check_against_step_path, _mixed, _model, _shortlist, _targets

pytestmark = pytest.mark.gpu
SCORE_CHUNK = 16384  # rows of the scoring pass's output stage per launch (engine.cu, kScoreChunk)


@pytest.fixture(scope="module")
def tiny(gpu_ctx, tiny_model):
    m = capi.Model(gpu_ctx, open(tiny_model[0], "rb").read())
    yield m
    m.close()


# the step path runs to the longest target only on models that never choose EOS (test_gpu_score.py, NO_EOS_BIAS)
@pytest.fixture(scope="module")
def tiny_no_eos(gpu_ctx, tmp_path_factory):
    m = _model(gpu_ctx, tmp_path_factory, synth.TINY, 1234, NO_EOS_BIAS)
    yield m
    m.close()


@pytest.fixture(scope="module")
def base_no_eos(gpu_ctx, tmp_path_factory):
    m = _model(gpu_ctx, tmp_path_factory, synth.BASE, 77, NO_EOS_BIAS)
    yield m
    m.close()


# ---------------------------------------------------------------- padded positions are computed and discarded
@pytest.mark.parametrize("model,src_len,tgt_lens", [
    ("tiny", (3, 9), _mixed(256) + [31, 63, 65]),
    ("tiny", (560, 600), [700, 1, 33, 65]),
    ("base_no_eos", (401, 460), [300, 1, 33, 65]),
], ids=["tiny-3-9", "tiny-560-600", "base-401-460"])
def test_scores_do_not_depend_on_longer_targets_in_the_batch(request, model, src_len, tgt_lens):
    """Full vocabulary only: a shortlist depends on the words of the whole batch."""
    m = request.getfixturevalue(model)
    m.set_max_length(1024)
    try:
        n = len(tgt_lens)
        sources = synth.make_sentences(n, src_len, seed=201 + src_len[0])
        targets = _targets(n, tgt_lens, seed=202)
        batch, st = m.score(sources, targets, max_words=BIG, want_alignments=True)
        assert st["batches"] == 1
        for i in range(n):
            alone, sa = m.score([sources[i]], [targets[i]], max_words=BIG, want_alignments=True)
            assert np.array_equal(batch[i].view(np.uint32), alone[0].view(np.uint32)), f"scores of sentence {i}"
            assert np.array_equal(st["alignments"][i].view(np.uint32), sa["alignments"][0].view(np.uint32)), f"alignment {i}"
    finally:
        m.set_max_length(256)


# ---------------------------------------------------------------- output rows in more than one chunk
@pytest.mark.parametrize("model,use_sl", [("tiny_no_eos", False), ("tiny_no_eos", True), ("base_no_eos", False)],
                         ids=["tiny-full", "tiny-shortlist", "base-full"])
def test_output_rows_in_two_chunks_match_step_path(request, shortlist_assets, model, use_sl):
    """600 sentences x 33 target positions: 19800 rows, a full chunk and a last one of 3416 rows (not a multiple of
    128).  Targets of 28-33 words, so padded positions sit in both chunks."""
    m = request.getfixturevalue(model)
    sources = synth.make_sentences(600, (4, 12), seed=211)
    sl = _shortlist(sources, shortlist_assets) if use_sl else None
    targets = _targets(600, [28, 29, 30, 31, 32, 33], seed=212, words=sl)
    M = len(targets) * max(len(t) for t in targets)
    assert M > SCORE_CHUNK and M % SCORE_CHUNK % 128 != 0
    _check_against_step_path(m, sources, targets, shortlist_assets, sl)


def test_headline_batch_matches_step_path(tiny, shortlist_assets):
    """tiny11 + shortlist, 4096 sentences of 32 tokens, their greedy translations as the targets (EOS included):
    4096 x 48 rows, twelve output chunks."""
    sources = synth.make_sentences(4096, 32, seed=1000)
    sl_bin = open(shortlist_assets[0], "rb").read()
    outs, st = tiny.translate(sources, max_words=BIG, shortlist_bin=sl_bin)
    assert st["batches"] == 1
    M = len(outs) * max(len(o) for o in outs)
    assert -(-M // SCORE_CHUNK) >= 12
    _check_against_step_path(tiny, sources, outs, shortlist_assets, _shortlist(sources, shortlist_assets))
