"""GPU: scoring given translations (slimt_b200_score, the time-parallel teacher-forced decoder).

The score of target token t_j is y[c] - LSE(y) over the logits y of the decoder fed the zero embedding at j = 0 and
t_{j-1} after that.  Checked against a float64 log-softmax over the oracle's logits at every position, bit for bit
against the step path (model_forward with forced + token_scores) on every route, and in round trips with
slimt_b200_translate (scores and alignments) and slimt_b200_translate_sampled."""
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
    """Oracle.encode, then Oracle.step with the forced words for exactly T_target steps (no early stop)."""
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
    prev = None
    for j in range(Tt):
        logits, _, _ = orc.step(enc, mask, states, prev, shortlist)
        out[:, j] = _log_softmax_at(logits.reshape(B, -1), _cols(tg[:, j], shortlist))
        prev = tg[:, j]
    return [out[b, :len(t)] for b, t in enumerate(targets)]


def _targets(n, lengths, seed, eos_every=0):
    rng = np.random.default_rng(seed)
    outs = []
    for i in range(n):
        L = int(lengths[i % len(lengths)])
        t = rng.integers(1, 32000, size=L).astype(np.uint32)
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


@pytest.fixture(scope="module")
def base(gpu_ctx, tmp_path_factory):
    path = str(tmp_path_factory.mktemp("model") / "base.bin")
    synth.write_model(path, synth.make_params(synth.BASE, seed=77))
    m = capi.Model(gpu_ctx, open(path, "rb").read())
    yield m
    m.close()


# ---------------------------------------------------------------- 1. against the oracle at every position
@pytest.mark.parametrize("use_sl", [False, True], ids=["full", "shortlist"])
def test_scores_match_oracle_every_position(tiny, shortlist_assets, use_sl):
    m, items = tiny
    sources = synth.make_sentences(5, (3, 9), seed=31)
    # targets longer than 1.5 x the source, with EOS in mid-target
    targets = _targets(5, [int(1.5 * len(s)) + 4 for s in sources], seed=32, eos_every=1)
    sl_bin = open(shortlist_assets[0], "rb").read() if use_sl else None
    got, st = m.score(sources, targets, max_words=BIG, shortlist_bin=sl_bin)
    assert st["batches"] == 1
    want = _oracle_scores(items, sources, targets, _shortlist(sources, shortlist_assets) if use_sl else None)
    for b in range(len(targets)):
        assert got[b].shape == (len(targets[b]),)
        fin = np.isfinite(want[b])
        assert np.array_equal(fin, np.isfinite(got[b]))
        assert np.abs(got[b][fin] - want[b][fin]).max() <= TOL


# ---------------------------------------------------------------- 2. bit-identical to the step path
def _step_path(m, sources, targets, shortlist):
    """model_forward with forced = the targets and token_scores: (scores [steps][B], steps executed)."""
    tokens, lengths = util.pad_batch(sources)
    B, T = tokens.shape
    max_steps = max(1, int(np.float32(1.5) * np.float32(T)))
    forced = np.zeros((max_steps, B), dtype=np.uint32)
    for b, t in enumerate(targets):
        n = min(len(t), max_steps)
        forced[:n, b] = t[:n]
    out = m.forward(tokens, lengths, shortlist=shortlist, forced=forced, want_scores=True)
    return out["scores"], out["steps"]


def _check_against_step_path(m, sources, targets, shortlist_assets, use_sl):
    sl_bin = open(shortlist_assets[0], "rb").read() if use_sl else None
    got, st = m.score(sources, targets, max_words=BIG, shortlist_bin=sl_bin)
    assert st["batches"] == 1
    ref, steps = _step_path(m, sources, targets, _shortlist(sources, shortlist_assets) if use_sl else None)
    compared = 0
    for b, t in enumerate(targets):
        n = min(len(t), steps)
        assert np.array_equal(got[b][:n].view(np.uint32), ref[:n, b].view(np.uint32)), f"sentence {b}"
        compared += n
    assert compared > 0


@pytest.mark.parametrize("use_sl", [False, True], ids=["full", "shortlist"])
@pytest.mark.parametrize("src_len", [(3, 32), (33, 64), (65, 256), (257, 300), (560, 600)],
                         ids=["le32", "33-64", "65-256", "257-300", "560-600"])
def test_bit_identical_to_step_path_tiny(tiny, shortlist_assets, src_len, use_sl):
    m, _ = tiny
    m.set_max_length(1024)
    try:
        sources = synth.make_sentences(4, src_len, seed=41 + src_len[0])
        targets = _targets(4, [7, 30, 12, 45], seed=42)
        _check_against_step_path(m, sources, targets, shortlist_assets, use_sl)
    finally:
        m.set_max_length(256)


@pytest.mark.parametrize("use_sl", [False, True], ids=["full", "shortlist"])
@pytest.mark.parametrize("src_len", [(3, 32), (65, 200)], ids=["le32", "65-256"])
def test_bit_identical_to_step_path_base(base, shortlist_assets, src_len, use_sl):
    sources = synth.make_sentences(4, src_len, seed=51)
    targets = _targets(4, [9, 20, 33, 5], seed=52)
    _check_against_step_path(base, sources, targets, shortlist_assets, use_sl)


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
