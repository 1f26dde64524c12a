"""GPU: per-token scores (log-probabilities) of a translation.  score[s][b] = y[c] - log sum_n exp(y[n]) over the step's
logits y (the shortlist's columns or the vocabulary's), c the greedy choice or the forced word's column.  The
reference values are float64 log_softmax over the oracle's logits; the fused scores GEMM must leave the tokens as they
are and agree bit for bit with the logits-tap route in exact mode."""
import numpy as np
import pytest

import sb_testutil as util
from oracle import slimt_oracle as so
from slimt_b200 import capi, synth
from test_gpu_out_fallback import _write_fallback_model

pytestmark = pytest.mark.gpu
TOL = 1e-4  # nats


def _log_softmax_at(logits, cols):
    """float64 log_softmax of each row of logits [B][N] at cols [B] (-1: -inf)."""
    L = np.asarray(logits, dtype=np.float64)
    m = L.max(axis=1)
    lse = m + np.log(np.exp(L - m[:, None]).sum(axis=1))
    out = np.full(L.shape[0], -np.inf)
    ok = cols >= 0
    out[ok] = L[ok, cols[ok]] - lse[ok]
    return out


def _ref_scores(ref, shortlist=None, forced=None):
    """[steps][B] reference scores from an oracle forward(keep=True)."""
    rows = []
    for s, L in enumerate(ref["logits"]):
        words = ref["step_tokens"][s] if forced is None else forced[s]
        if shortlist is None:
            cols = np.asarray(words, dtype=np.int64)
        else:
            pos = np.searchsorted(shortlist, words)
            hit = (pos < len(shortlist)) & (shortlist[np.minimum(pos, len(shortlist) - 1)] == words)
            cols = np.where(hit, pos, -1)
        rows.append(_log_softmax_at(L, cols))
    return np.stack(rows)


def _batch(n, length, seed):
    sents = synth.make_sentences(n, length, seed=seed)
    tokens, lengths = util.pad_batch(sents)
    return sents, tokens, lengths


@pytest.fixture(scope="module")
def tiny(gpu_ctx, tiny_model):
    path, items = tiny_model
    m = capi.Model(gpu_ctx, open(path, "rb").read())
    yield m, items, path
    m.close()


def _shortlist(sents, shortlist_assets):
    _, (fr, offs, lists) = shortlist_assets
    return so.shortlist_generate(np.concatenate(sents), fr, offs, lists, 32000)


@pytest.mark.parametrize("use_sl", [False, True], ids=["full", "shortlist"])
def test_exact_scores_match_reference(tiny, shortlist_assets, use_sl):
    m, items, _ = tiny
    sents, tokens, lengths = _batch(24, (2, 20), seed=21)
    sl = _shortlist(sents, shortlist_assets) if use_sl else None
    ref = so.Oracle(items).forward(tokens, lengths, shortlist=sl, keep=True)
    plain = m.forward(tokens, lengths, shortlist=sl)
    out = m.forward(tokens, lengths, shortlist=sl, want_scores=True)
    assert out["steps"] == plain["steps"] == len(ref["step_tokens"])
    assert np.array_equal(out["step_tokens"], plain["step_tokens"])
    assert np.array_equal(out["step_tokens"], ref["step_tokens"])
    want = _ref_scores(ref, sl)
    assert out["scores"].shape == want.shape
    assert np.abs(out["scores"] - want).max() <= TOL
    assert (out["scores"] <= 1e-6).all()


@pytest.mark.parametrize("fast", [False, True], ids=["exact", "tolerance"])
@pytest.mark.parametrize("use_sl", [False, True], ids=["full", "shortlist"])
def test_scores_route_equals_tap_route(tiny_model, shortlist_assets, fast, use_sl):
    path, _ = tiny_model
    ctx = capi.Context(0)
    ctx.set_math(fast)
    m = capi.Model(ctx, open(path, "rb").read())
    sents, tokens, lengths = _batch(16, (3, 24), seed=5)
    sl = _shortlist(sents, shortlist_assets) if use_sl else None
    fused = m.forward(tokens, lengths, shortlist=sl, want_scores=True)
    tap = m.forward(tokens, lengths, shortlist=sl, want_scores=True, want_logits=True)
    assert np.array_equal(fused["step_tokens"], tap["step_tokens"])
    if not fast:
        assert np.array_equal(fused["scores"], tap["scores"])
    cols = [tap["logits"][s].argmax(axis=1) for s in range(tap["steps"])]
    want = np.stack([_log_softmax_at(tap["logits"][s], cols[s]) for s in range(tap["steps"])])
    assert np.abs(fused["scores"] - want).max() <= TOL
    assert np.abs(tap["scores"] - want).max() <= TOL
    m.close()
    ctx.close()


def test_teacher_forcing_outside_the_shortlist(tiny, shortlist_assets):
    m, items, _ = tiny
    sents, tokens, lengths = _batch(16, (3, 20), seed=33)
    sl = _shortlist(sents, shortlist_assets)
    steps = int(np.float32(1.5) * np.float32(tokens.shape[1]))
    rng = np.random.RandomState(4)
    inside = sl[rng.randint(0, len(sl), size=(steps, len(sents)))]
    anywhere = rng.randint(1, 32000, size=(steps, len(sents)))
    forced = np.where(rng.rand(steps, len(sents)) < 0.5, inside, anywhere).astype(np.uint32)
    ref = so.Oracle(items).forward(tokens, lengths, shortlist=sl, forced=forced, keep=True)
    out = m.forward(tokens, lengths, shortlist=sl, forced=forced, want_scores=True)
    assert np.array_equal(out["step_tokens"], ref["step_tokens"])
    want = _ref_scores(ref, sl, forced)
    got = out["scores"]
    outside = np.isneginf(want)
    assert outside.any() and (~outside).any()
    assert np.array_equal(np.isneginf(got), outside)
    assert np.abs(got[~outside] - want[~outside]).max() <= TOL
    # without a shortlist every forced word is a column
    ref_full = so.Oracle(items).forward(tokens, lengths, forced=forced, keep=True)
    full = m.forward(tokens, lengths, forced=forced, want_scores=True)
    assert np.abs(full["scores"] - _ref_scores(ref_full, None, forced)).max() <= TOL


@pytest.fixture(scope="module")
def fallback_model(tmp_path_factory):
    return _write_fallback_model(tmp_path_factory, synth.TINY, "tiny11_scores")


@pytest.fixture(scope="module")
def base_model(tmp_path_factory):
    path = str(tmp_path_factory.mktemp("model") / "base_scores.bin")
    synth.write_model(path, synth.make_params(synth.BASE, seed=1234))
    return path, synth.read_model(path)


@pytest.mark.parametrize("which", ["bound_filter", "base"])
def test_other_models(gpu_ctx, shortlist_assets, fallback_model, base_model, which):
    """A model whose offsets exceed the digits (bound filter, K = 256) and the base model (K = 512)."""
    path, items = fallback_model if which == "bound_filter" else base_model
    m = capi.Model(gpu_ctx, open(path, "rb").read())
    sents, tokens, lengths = _batch(8, (2, 12), seed=17)
    orc = so.Oracle(items)
    for sl in (None, _shortlist(sents, shortlist_assets)):
        ref = orc.forward(tokens, lengths, shortlist=sl, keep=True)
        out = m.forward(tokens, lengths, shortlist=sl, want_scores=True)
        assert np.array_equal(out["step_tokens"], ref["step_tokens"])
        assert np.abs(out["scores"] - _ref_scores(ref, sl)).max() <= TOL
    m.close()


def test_determinism(gpu_ctx, tiny, shortlist_assets):
    m, _, _ = tiny
    sents, tokens, lengths = _batch(12, (3, 18), seed=8)
    sl = _shortlist(sents, shortlist_assets)
    a = m.forward(tokens, lengths, shortlist=sl, want_scores=True)
    b = m.forward(tokens, lengths, shortlist=sl, want_scores=True)
    assert np.array_equal(a["scores"], b["scores"])
    # one sentence, two sets of companions, same batch width, full vocabulary
    pool = synth.make_sentences(9, (2, 10), seed=44)
    first = synth.make_sentences(1, (14, 14), seed=45)[0]
    runs = []
    for companions in (pool[:4], pool[4:8]):
        t, l = util.pad_batch([first] + list(companions))
        assert t.shape[1] == len(first)
        runs.append(m.forward(t, l, want_scores=True))
    n = min(runs[0]["steps"], runs[1]["steps"])
    assert np.array_equal(runs[0]["step_tokens"][:n, 0], runs[1]["step_tokens"][:n, 0])
    assert np.array_equal(runs[0]["scores"][:n, 0], runs[1]["scores"][:n, 0])
    # device-resident input and output
    B, T = tokens.shape
    max_steps = int(np.float32(1.5) * np.float32(T))
    d_tok, d_len, d_sl = gpu_ctx.to_device(tokens), gpu_ctx.to_device(lengths), gpu_ctx.to_device(sl)
    d_steps, d_scores = gpu_ctx.dev_alloc(4 * max_steps * B), gpu_ctx.dev_alloc(4 * max_steps * B)
    steps, _ = m.forward_resident(d_tok, d_len, B, T, d_steps, d_shortlist=d_sl, n_shortlist=len(sl), d_scores=d_scores)
    dev_steps = gpu_ctx.from_device(d_steps, (max_steps, B), np.uint32)[:steps]
    dev_scores = gpu_ctx.from_device(d_scores, (max_steps, B), np.float32)[:steps]
    for p in (d_tok, d_len, d_sl, d_steps, d_scores):
        gpu_ctx.dev_free(p)
    assert steps == a["steps"]
    assert np.array_equal(dev_steps, a["step_tokens"])
    assert np.array_equal(dev_scores, a["scores"])


@pytest.mark.parametrize("use_sl", [False, True], ids=["full", "shortlist"])
def test_launch_counts(gpu_ctx, tiny, shortlist_assets, use_sl):
    """Fused route: the parent's launches plus one score_step per executed step, minus the shortlist's table build."""
    m, _, _ = tiny
    sents, tokens, lengths = _batch(32, (3, 20), seed=61)
    sl = _shortlist(sents, shortlist_assets) if use_sl else None

    def run(**kw):
        gpu_ctx.profile(True)
        l0 = gpu_ctx.launches()
        m.forward(tokens, lengths, shortlist=sl, **kw)
        n = gpu_ctx.launches() - l0
        prof = {r["name"]: r["launches"] for r in gpu_ctx.profile_read()}
        gpu_ctx.profile(False)
        return n, prof

    n0, p0 = run()
    n1, p1 = run(want_scores=True)
    executed = p0["dec_gemm_out_argmax"]
    assert p1["dec_gemm_out_scores"] == executed and p1["score_step"] == executed
    assert "dec_gemm_out_argmax" not in p1 and "out_bounds" not in p1
    assert n1 == n0 + executed - (1 if use_sl else 0)


def test_service_scores(gpu_ctx, tiny_model, shortlist_assets, monkeypatch):
    path, _ = tiny_model
    sl_path, _ = shortlist_assets
    sl_bin = open(sl_path, "rb").read()
    model_bin = open(path, "rb").read()
    monkeypatch.setenv("SLIMT_B200_LANES", "2")
    r1, r2 = capi.Model(gpu_ctx, model_bin), capi.Model(gpu_ctx, model_bin)
    sents = synth.make_sentences(60, (2, 24), seed=71)
    max_words = 160
    outs, st = r1.translate(sents, max_words=max_words, shortlist_bin=sl_bin, replicas=[r1, r2], want_scores=True)
    plain, _ = r1.translate(sents, max_words=max_words, shortlist_bin=sl_bin, replicas=[r1, r2])
    assert [o.tolist() for o in outs] == [o.tolist() for o in plain]
    assert [len(s) for s in st["scores"]] == [len(o) for o in outs]
    assert st["batches"] > 2
    for ids, width in capi.batcher_plan([len(s) for s in sents], max_words):
        batch = [sents[i] for i in ids]
        tokens, lengths = util.pad_batch(batch)
        assert tokens.shape[1] == width
        sl = capi.shortlist_generate(sl_bin, np.concatenate(batch), 32000)
        fwd = r1.forward(tokens, lengths, shortlist=sl, want_scores=True)
        for r, i in enumerate(ids):
            assert np.array_equal(st["scores"][i], fwd["scores"][:len(outs[i]), r])
    # ragged like out_tokens: a capacity too small for the tokens fails cleanly
    offsets = np.zeros(len(sents) + 1, dtype=np.uint64)
    offsets[1:] = np.cumsum([len(s) for s in sents])
    flat = np.concatenate(sents).astype(np.uint32)
    with pytest.raises(RuntimeError, match="capacity too small"):
        r1.translate_flat(flat, offsets, max_words, shortlist_bin=sl_bin, out_tokens=np.zeros(4, np.uint32),
                          want_scores=True)
    r1.close()
    r2.close()
