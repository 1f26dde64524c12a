"""GPU: scoring given translations (slimt_b200_score, the time-parallel teacher-forced decoder).

The score of target token t_j is y[c] - LSE(y) over the logits y of the decoder fed the zero embedding at j = 0 and
t_{j-1} after that.  Checked against a float64 log-softmax over the oracle's logits at every position, bit for bit
against the step path (model_forward with forced + token_scores + alignment, run to the longest target) at every target
position on every route, and in round trips with slimt_b200_translate (scores and alignments) and
slimt_b200_translate_sampled.  test_gpu_score_edges.py holds the batch-level cases (padding, output row chunks)."""
import numpy as np
import pytest

import sb_testutil as util
from oracle import slimt_oracle as so
from slimt_b200 import capi, synth

pytestmark = pytest.mark.gpu
TOL = 1e-4  # nats: test_gpu_scores.py's bar against the oracle
BIG = 1 << 20  # max_words large enough for one batch


def _log_softmax_at(logits, cols):
    L = np.asarray(logits, dtype=np.float64)
    m = L.max(axis=1)
    lse = m + np.log(np.exp(L - m[:, None]).sum(axis=1))
    out = np.full(L.shape[0], -np.inf)
    ok = cols >= 0
    out[ok] = L[ok, cols[ok]] - lse[ok]
    return out


def _cols(words, shortlist):
    words = np.asarray(words, dtype=np.int64)
    if shortlist is None:
        return words
    pos = np.searchsorted(shortlist, words)
    hit = (pos < len(shortlist)) & (shortlist[np.minimum(pos, len(shortlist) - 1)] == words)
    return np.where(hit, pos, -1)


def _oracle_scores(items, sources, targets, shortlist=None):
    """Oracle.encode, then Oracle.step with the forced words for exactly T_target steps (no early stop).  Returns each
    target's log-probabilities and its alignment: head 0 of the last layer's attention over the sentence's tokens."""
    orc = so.Oracle(items)
    tokens, lengths = util.pad_batch(sources)
    B, T = tokens.shape
    mask01 = (np.arange(T)[None, :] < np.asarray(lengths)[:, None]).astype(np.float32)
    mask = ((np.float32(1) - mask01) * np.float32(-99999999.0)).astype(np.float32)
    enc = orc.encode(tokens, mask)
    Tt = max(len(t) for t in targets)
    tg = np.zeros((B, Tt), dtype=np.uint32)
    for b, t in enumerate(targets):
        tg[b, :len(t)] = t
    states = [np.zeros((B, 1, orc.W.E), dtype=np.float32) for _ in range(orc.Ld)]
    out = np.zeros((B, Tt))
    align = np.zeros((B, Tt, T), dtype=np.float32)
    prev = None
    for j in range(Tt):
        logits, attn, _ = orc.step(enc, mask, states, prev, shortlist)
        out[:, j] = _log_softmax_at(logits.reshape(B, -1), _cols(tg[:, j], shortlist))
        align[:, j] = attn[:, 0, 0, :]
        prev = tg[:, j]
    return ([out[b, :len(t)] for b, t in enumerate(targets)],
            [align[b, :len(t), :len(sources[b])] for b, t in enumerate(targets)])


def _targets(n, lengths, seed, eos_every=0, words=None):
    """n targets, the i-th of lengths[i % len(lengths)] words: uniform over the vocabulary without EOS, or over `words`
    without EOS (a shortlist, so that the scores are finite rather than -inf for words outside the output columns)."""
    rng = np.random.default_rng(seed)
    pool = None if words is None else np.asarray(words, dtype=np.uint32)[np.asarray(words) != 0]
    outs = []
    for i in range(n):
        L = int(lengths[i % len(lengths)])
        if pool is None:
            t = rng.integers(1, 32000, size=L).astype(np.uint32)
        else:
            t = pool[rng.integers(0, len(pool), size=L)]
        if eos_every and L > 2:
            t[L // 2] = 0  # EOS in mid-target: scored like any other word, scoring goes on
        outs.append(t)
    return outs


def _shortlist(sents, shortlist_assets):
    _, (fr, offs, lists) = shortlist_assets
    return so.shortlist_generate(np.concatenate(sents), fr, offs, lists, 32000)


@pytest.fixture(scope="module")
def tiny(gpu_ctx, tiny_model):
    path, items = tiny_model
    m = capi.Model(gpu_ctx, open(path, "rb").read())
    yield m, items
    m.close()


@pytest.fixture(scope="module")
def eos(gpu_ctx, eos_model):
    path, items = eos_model
    m = capi.Model(gpu_ctx, open(path, "rb").read())
    yield m, items
    m.close()


# The step path's decode loop ends once every sentence's greedy choice has been EOS: a forced word replaces only the
# next input, as in the reference (Model.cc:127-161).  Models with this output bias on EOS (about 30 nats below the best
# logit) never choose it, so the step path runs to its step limit and every target position can be compared.
NO_EOS_BIAS = -30.0


def _model(ctx, tmp_path_factory, dims, seed, eos_bias):
    path = str(tmp_path_factory.mktemp("model") / "model.bin")
    synth.write_model(path, synth.make_params(dims, seed=seed, eos_bias=eos_bias))
    return capi.Model(ctx, open(path, "rb").read())


@pytest.fixture(scope="module")
def tiny_no_eos(gpu_ctx, tmp_path_factory):
    """tiny11 with the weights of conftest's tiny_model, but NO_EOS_BIAS."""
    m = _model(gpu_ctx, tmp_path_factory, synth.TINY, 1234, NO_EOS_BIAS)
    yield m
    m.close()


@pytest.fixture(scope="module")
def base(gpu_ctx, tmp_path_factory):
    m = _model(gpu_ctx, tmp_path_factory, synth.BASE, 77, NO_EOS_BIAS)
    yield m
    m.close()


# ---------------------------------------------------------------- 1. against the oracle at every position
@pytest.mark.parametrize("use_sl,long_targets", [(False, False), (True, False), (False, True), (True, True)],
                         ids=["full", "shortlist", "60-100-full", "60-100-shortlist"])
def test_scores_match_oracle_every_position(tiny, shortlist_assets, use_sl, long_targets):
    m, items = tiny
    n = 4 if long_targets else 5  # the oracle steps the whole batch once per target position: keep it small
    sources = synth.make_sentences(n, (3, 9), seed=31)
    sl = _shortlist(sources, shortlist_assets) if use_sl else None
    # targets longer than 1.5 x the source, with EOS in mid-target; the long ones span two 32-position scan tiles and
    # one or two 64-query blocks of the cross-attention
    lengths = [60, 65, 97, 100] if long_targets else [int(1.5 * len(s)) + 4 for s in sources]
    targets = _targets(n, lengths, seed=32, eos_every=1, words=sl)
    sl_bin = open(shortlist_assets[0], "rb").read() if use_sl else None
    got, st = m.score(sources, targets, max_words=BIG, shortlist_bin=sl_bin, want_alignments=True)
    assert st["batches"] == 1
    want, want_al = _oracle_scores(items, sources, targets, sl)
    for b in range(len(targets)):
        assert got[b].shape == (len(targets[b]),)
        fin = np.isfinite(want[b])
        assert fin.all()
        assert np.array_equal(fin, np.isfinite(got[b]))
        assert np.abs(got[b][fin] - want[b][fin]).max() <= TOL, f"sentence {b}"
        # the alignment is bit-exact against the oracle's attention, as on the step path (test_gpu_long_sentences.py)
        assert np.array_equal(st["alignments"][b], want_al[b]), f"alignment of sentence {b}"


# ---------------------------------------------------------------- 2. bit-identical to the step path
def _step_path(m, sources, targets, shortlist):
    """model_forward with forced = the targets, token_scores and alignments, with a limit factor that lets it execute
    every position of the longest target: (scores [steps][B], alignment [steps][B][T])."""
    tokens, lengths = util.pad_batch(sources)
    B, T = tokens.shape
    longest = max(len(t) for t in targets)
    lf = max(1.5, (longest + 0.5) / T)
    max_steps = max(1, int(np.float32(lf) * np.float32(T)))
    assert max_steps >= longest
    forced = np.zeros((max_steps, B), dtype=np.uint32)  # the words after a target are fed but never compared
    for b, t in enumerate(targets):
        forced[:len(t), b] = t
    out = m.forward(tokens, lengths, limit_factor=lf, shortlist=shortlist, forced=forced, want_scores=True,
                    want_alignment=True)
    assert out["steps"] >= longest, "every sentence chose EOS before the longest target ended (NO_EOS_BIAS)"
    return out["scores"], out["alignment"]


def _check_against_step_path(m, sources, targets, shortlist_assets, shortlist):
    """slimt_b200_score of one batch against the step path on the same padded batch, bit for bit at every target
    position: scores, and alignments over each sentence's own tokens.  shortlist: the batch's (_shortlist), or None
    for the full vocabulary."""
    sl_bin = open(shortlist_assets[0], "rb").read() if shortlist is not None else None
    got, st = m.score(sources, targets, max_words=BIG, shortlist_bin=sl_bin, want_alignments=True)
    assert st["batches"] == 1
    ref, ref_al = _step_path(m, sources, targets, shortlist)
    for b, t in enumerate(targets):
        n, L = len(t), len(sources[b])
        assert np.array_equal(got[b].view(np.uint32), ref[:n, b].view(np.uint32)), f"scores of sentence {b}"
        assert np.array_equal(st["alignments"][b].view(np.uint32), ref_al[:n, b, :L].view(np.uint32)), f"alignment {b}"
    # the targets are among the output columns: no position compares -inf with -inf alone
    assert np.isfinite(np.concatenate(got)).all()


def _mixed(longest):
    """Target lengths of one batch: `longest` (the padded width) beside shorter targets, so that padded positions
    share every tile with live ones."""
    return [longest] + [n for n in (1, 32, 33, 64, 97) if n < longest]


def _step_path_case(m, shortlist_assets, use_sl, src_len, tgt_lens, seed):
    n = max(4, len(tgt_lens))
    sources = synth.make_sentences(n, src_len, seed=seed)
    sl = _shortlist(sources, shortlist_assets) if use_sl else None
    targets = _targets(n, tgt_lens, seed=seed + 1, words=sl)
    _check_against_step_path(m, sources, targets, shortlist_assets, sl)


# source lengths x target lengths of one batch.  Sources of 3-9 tokens with targets far beyond 1.5 x the source, target
# widths on both sides of the scan's 32-position tiles and the tiled kernel's 64-query blocks; 560-600 tokens: the long
# kernel (head size 32, 32-query blocks) with targets up to 700.
TINY_CASES = [((3, 32), [7, 30, 12, 45]), ((33, 64), [7, 30, 12, 45]), ((65, 256), [7, 30, 12, 45]),
              ((257, 300), [7, 30, 12, 45]), ((560, 600), [7, 30, 12, 45])]
TINY_IDS = ["le32", "33-64", "65-256", "257-300", "560-600"]
for _n in (1, 31, 32, 33, 63, 64, 65, 97, 256):
    TINY_CASES.append(((3, 9), _mixed(_n)))
    TINY_IDS.append(f"3-9-to-{_n}")
for _n in (33, 65, 700):
    TINY_CASES.append(((560, 600), _mixed(_n)))
    TINY_IDS.append(f"560-600-to-{_n}")


@pytest.mark.parametrize("use_sl", [False, True], ids=["full", "shortlist"])
@pytest.mark.parametrize("src_len,tgt_lens", TINY_CASES, ids=TINY_IDS)
def test_bit_identical_to_step_path_tiny(tiny_no_eos, shortlist_assets, src_len, tgt_lens, use_sl):
    m = tiny_no_eos
    m.set_max_length(1024)
    try:
        _step_path_case(m, shortlist_assets, use_sl, src_len, tgt_lens, seed=41 + src_len[0] + 1000 * tgt_lens[0])
    finally:
        m.set_max_length(256)


# base (E = 512, head size 64): 401-460 source tokens take the long kernel; 3-9 with long targets give the scan many tiles
BASE_CASES = [((3, 32), [9, 20, 33, 5]), ((65, 200), [9, 20, 33, 5])]
BASE_IDS = ["le32", "65-256"]
for _n in (33, 65, 300):
    BASE_CASES.append(((401, 460), _mixed(_n)))
    BASE_IDS.append(f"401-460-to-{_n}")
for _n in (33, 65, 256):
    BASE_CASES.append(((3, 9), _mixed(_n)))
    BASE_IDS.append(f"3-9-to-{_n}")


@pytest.mark.parametrize("use_sl", [False, True], ids=["full", "shortlist"])
@pytest.mark.parametrize("src_len,tgt_lens", BASE_CASES, ids=BASE_IDS)
def test_bit_identical_to_step_path_base(base, shortlist_assets, src_len, tgt_lens, use_sl):
    base.set_max_length(1024)
    try:
        _step_path_case(base, shortlist_assets, use_sl, src_len, tgt_lens, seed=51 + src_len[0] + 1000 * tgt_lens[0])
    finally:
        base.set_max_length(256)


# ---------------------------------------------------------------- 3. round trips
@pytest.mark.parametrize("use_sl", [False, True], ids=["full", "shortlist"])
def test_round_trip_translate(eos, shortlist_assets, use_sl):
    m, _ = eos
    sources = synth.make_sentences(40, (2, 20), seed=61)
    sl_bin = open(shortlist_assets[0], "rb").read() if use_sl else None
    outs, tst = m.translate(sources, max_words=128, shortlist_bin=sl_bin, want_scores=True, want_alignments=True)
    got, sst = m.score(sources, outs, max_words=128, shortlist_bin=sl_bin, want_alignments=True)
    assert sst["batches"] == tst["batches"] > 1
    for i in range(len(sources)):
        assert np.array_equal(got[i].view(np.uint32), tst["scores"][i].view(np.uint32)), f"scores of sentence {i}"
        assert np.array_equal(sst["alignments"][i].view(np.uint32), tst["alignments"][i].view(np.uint32)), f"alignment {i}"


def test_round_trip_sampled(eos, shortlist_assets):
    m, _ = eos
    sources = synth.make_sentences(24, (2, 16), seed=71)
    sl_bin = open(shortlist_assets[0], "rb").read()
    outs, tst = m.translate(sources, max_words=96, shortlist_bin=sl_bin, want_scores=True,
                            sampling={"temperature": 1.0, "seed": 5})
    got, _ = m.score(sources, outs, max_words=96, shortlist_bin=sl_bin)
    for i in range(len(sources)):
        assert np.array_equal(got[i].view(np.uint32), tst["scores"][i].view(np.uint32)), f"sentence {i}"


# ---------------------------------------------------------------- 4. service
def test_two_replicas_and_fast_context_give_the_same_bits(gpu_ctx, tiny_model, tiny, shortlist_assets):
    m, _ = tiny
    sources = synth.make_sentences(60, (2, 18), seed=81)
    targets = _targets(60, [0, 5, 17, 26], seed=82)
    sl_bin = open(shortlist_assets[0], "rb").read()
    one, st1 = m.score(sources, targets, max_words=64, shortlist_bin=sl_bin, want_alignments=True)
    assert st1["batches"] >= 4
    m2 = capi.Model(gpu_ctx, open(tiny_model[0], "rb").read())
    try:
        two, st2 = m.score(sources, targets, max_words=64, shortlist_bin=sl_bin, replicas=[m, m2], want_alignments=True)
    finally:
        m2.close()
    gpu_ctx.set_math(True)
    try:
        fast, _ = m.score(sources, targets, max_words=64, shortlist_bin=sl_bin)
    finally:
        gpu_ctx.set_math(False)
    for i in range(len(sources)):
        assert np.array_equal(one[i].view(np.uint32), two[i].view(np.uint32))
        assert np.array_equal(one[i].view(np.uint32), fast[i].view(np.uint32))
        assert np.array_equal(st1["alignments"][i], st2["alignments"][i])


def test_empty_targets(tiny, shortlist_assets):
    m, _ = tiny
    sources = synth.make_sentences(6, (3, 9), seed=91)
    targets = _targets(6, [0, 4, 0, 7, 3, 0], seed=92)
    got, st = m.score(sources, targets, max_words=BIG, want_alignments=True)
    for i, t in enumerate(targets):
        assert got[i].shape == (len(t),) and st["alignments"][i].shape == (len(t), len(sources[i]))
    ref, _ = m.score([sources[i] for i in (1, 3, 4)], [targets[i] for i in (1, 3, 4)], max_words=BIG)
    for k, i in enumerate((1, 3, 4)):
        assert np.array_equal(got[i], ref[k])
    none, st = m.score(sources, [np.zeros(0, np.uint32)] * 6, max_words=BIG)
    assert all(len(x) == 0 for x in none) and st["kernel_launches"] == 0


def test_errors_fail_cleanly_and_model_stays_usable(tiny):
    m, items = tiny
    sources = synth.make_sentences(4, (3, 9), seed=101)
    tokens, lengths = util.pad_batch(sources)
    before = m.forward(tokens, lengths)["step_tokens"]
    targets = _targets(4, [5], seed=102)
    bad_word = [t.copy() for t in targets]
    bad_word[2][1] = 32000
    with pytest.raises(RuntimeError, match="outside the vocabulary"):
        m.score(sources, bad_word, max_words=BIG)
    with pytest.raises(RuntimeError, match="exceeds the supported maximum"):
        m.score(sources, _targets(4, [5, 300], seed=103), max_words=BIG)
    with pytest.raises(RuntimeError, match="exceeds the supported maximum"):
        m.score([np.arange(1, 300, dtype=np.uint32)] + sources[1:], targets, max_words=BIG)
    tok = np.concatenate(sources)
    off = np.zeros(5, np.uint64)
    off[1:] = np.cumsum([len(s) for s in sources])
    tg = np.concatenate(targets)
    toff = np.zeros(5, np.uint64)
    toff[1:] = np.cumsum([len(t) for t in targets])
    with pytest.raises(RuntimeError, match="non-decreasing"):
        capi.score_flat([m], tok, off, tg, toff[[0, 2, 1, 3, 4]], max_words=BIG)
    with pytest.raises(RuntimeError, match="capacity too small"):
        capi.score_flat([m], tok, off, tg, toff, max_words=BIG, out_capacity=len(tg) - 1)
    with pytest.raises(RuntimeError, match="capacity too small"):
        capi.score_flat([m], tok, off, tg, toff, max_words=BIG, want_alignments=True, align_capacity=3)
    assert np.array_equal(m.forward(tokens, lengths)["step_tokens"], before)
    ok, _ = m.score(sources, targets, max_words=BIG)
    assert [len(x) for x in ok] == [len(t) for t in targets]


# ---------------------------------------------------------------- 5. time-parallel structure
def test_launches_do_not_grow_with_target_length(tiny, shortlist_assets):
    m, _ = tiny
    sources = synth.make_sentences(8, (4, 12), seed=111)
    sl_bin = open(shortlist_assets[0], "rb").read()
    _, s8 = m.score(sources, _targets(8, [8], seed=112), max_words=BIG, shortlist_bin=sl_bin)
    _, s64 = m.score(sources, _targets(8, [64], seed=113), max_words=BIG, shortlist_bin=sl_bin)
    assert s8["batches"] == s64["batches"] == 1
    assert s8["kernel_launches"] == s64["kernel_launches"]
