"""GPU: sampled decoding (include/slimt_b200.h, DESIGN §4.4b).  Each step's word is the first column whose cumulative
probability under softmax(fl32(y * inv_t)) exceeds the step's Philox uniform number u; the reference below recomputes
u in numpy and the CDF in float64 from the logits tap of the same call."""
import math

import numpy as np
import pytest
from scipy import stats

import sb_testutil as util
from oracle import slimt_oracle as so
from slimt_b200 import capi, synth
from test_sample_rng import uniform_np

pytestmark = pytest.mark.gpu
EPS = 1e-5   # CDF slack
TOL = 1e-4   # nats


@pytest.fixture(scope="module")
def models(gpu_ctx, tiny_model, eos_model):
    ms = {"tiny": capi.Model(gpu_ctx, open(tiny_model[0], "rb").read()),
          "eos": capi.Model(gpu_ctx, open(eos_model[0], "rb").read())}
    yield ms
    for m in ms.values():
        m.close()


@pytest.fixture(scope="module")
def fast_model(tiny_model):
    ctx = capi.Context(0)
    ctx.set_math(True)
    m = capi.Model(ctx, open(tiny_model[0], "rb").read())
    yield m
    m.close()
    ctx.close()


def _shortlist(sents, shortlist_assets):
    _, (fr, offs, lists) = shortlist_assets
    return so.shortlist_generate(np.concatenate(sents), fr, offs, lists, 32000)


def _inv_t(temperature):
    return np.float32(1.0 / float(np.float32(temperature)))


def _check_against_float64(out, temperature, seed, keys, sl):
    """Check 1 over every row of every executed step of a call made with want_logits and want_scores."""
    inv_t = _inv_t(temperature)
    B = out["step_tokens"].shape[1]
    keys = np.arange(B, dtype=np.uint64) if keys is None else np.asarray(keys, dtype=np.uint64)
    exact = 0
    for s in range(out["steps"]):
        z = (out["logits"][s].astype(np.float32) * inv_t).astype(np.float64)
        lse = z.max(axis=1) + np.log(np.exp(z - z.max(axis=1, keepdims=True)).sum(axis=1))
        F = np.cumsum(np.exp(z - lse[:, None]), axis=1)
        u = uniform_np(np.full(B, seed, dtype=np.uint64), keys, np.full(B, s, dtype=np.uint64)).astype(np.float64) * 2.0**-53
        words = out["step_tokens"][s].astype(np.int64)
        cols = words if sl is None else np.searchsorted(sl, words)
        if sl is not None:
            assert np.array_equal(sl[cols], words)
        r = np.arange(B)
        lo = np.where(cols > 0, F[r, np.maximum(cols - 1, 0)], 0.0)
        assert (lo - EPS <= u).all() and (u <= F[r, cols] + EPS).all(), s
        clear = np.abs(F - u[:, None]).min(axis=1) > EPS
        want = np.array([np.searchsorted(F[b], u[b], side="right") for b in range(B)])
        assert np.array_equal(cols[clear], want[clear]), s
        exact += int(clear.sum())
        sc = out["scores"][s].astype(np.float64)
        assert np.isfinite(sc).all()
        assert np.abs(sc - (z[r, cols] - lse)).max() <= TOL, s
    assert exact > 0


@pytest.mark.parametrize("temperature", [0.5, 1.0, 2.0])
@pytest.mark.parametrize("use_sl", [False, True], ids=["full", "shortlist"])
@pytest.mark.parametrize("which", ["tiny", "eos"])
def test_against_float64_and_routes(models, shortlist_assets, which, use_sl, temperature):
    m = models[which]
    sents = synth.make_sentences(24, (2, 16), seed=301)
    tokens, lengths = util.pad_batch(sents)
    sl = _shortlist(sents, shortlist_assets) if use_sl else None
    sp = {"temperature": temperature, "seed": 11}
    tap = m.forward(tokens, lengths, shortlist=sl, want_logits=True, want_scores=True, sampling=sp)
    _check_against_float64(tap, temperature, 11, None, sl)
    fused = m.forward(tokens, lengths, shortlist=sl, want_scores=True, sampling=sp)
    assert fused["steps"] == tap["steps"]
    assert np.array_equal(fused["step_tokens"], tap["step_tokens"])
    assert np.array_equal(fused["scores"], tap["scores"])
    # without scores the same words
    bare = m.forward(tokens, lengths, shortlist=sl, sampling=sp)
    assert np.array_equal(bare["step_tokens"], tap["step_tokens"])


@pytest.mark.parametrize("use_sl", [False, True], ids=["full", "shortlist"])
def test_tolerance_mode_against_its_tap(fast_model, shortlist_assets, use_sl):
    sents = synth.make_sentences(16, (3, 16), seed=302)
    tokens, lengths = util.pad_batch(sents)
    sl = _shortlist(sents, shortlist_assets) if use_sl else None
    sp = {"temperature": 0.8, "seed": 5, "keys": np.arange(100, 116, dtype=np.uint64)}
    tap = fast_model.forward(tokens, lengths, shortlist=sl, want_logits=True, want_scores=True, sampling=sp)
    _check_against_float64(tap, 0.8, 5, sp["keys"], sl)
    fused = fast_model.forward(tokens, lengths, shortlist=sl, want_logits=False, want_scores=True, sampling=sp)
    assert fused["steps"] >= 1 and np.isfinite(fused["scores"]).all()


def test_distribution_chi_square(models):
    m = models["tiny"]
    sent = synth.make_sentences(1, (8, 8), seed=303)[0]
    one_t, one_l = util.pad_batch([sent])
    y = m.forward(one_t, one_l, want_logits=True)["logits"][0][0]
    # the highest temperature at which 30 words hold 90 % of step 0's mass
    for temperature in (1.0, 0.5, 0.3, 0.2, 0.1, 0.05, 0.02):
        z = (y.astype(np.float32) * _inv_t(temperature)).astype(np.float64)
        p = np.exp(z - z.max())
        p /= p.sum()
        if np.sort(p)[-30:].sum() >= 0.9:
            break
    B = 4096
    tokens, lengths = np.tile(one_t, (B, 1)), np.tile(one_l, B)
    out = m.forward(tokens, lengths, limit_factor=0.01, sampling={"temperature": temperature, "seed": 2024})
    assert out["step_tokens"].shape[0] >= 1
    counts = np.bincount(out["step_tokens"][0].astype(np.int64), minlength=len(p))
    expected = B * p
    big = expected >= 5
    obs = np.append(counts[big], counts[~big].sum())
    exp = np.append(expected[big], expected[~big].sum())
    if exp[-1] < 5:  # fold a thin tail into the smallest category
        obs, exp = obs[:-1], exp[:-1]
        obs[-1] += counts[~big].sum()
        exp[-1] += expected[~big].sum()
    assert big.sum() >= 5
    assert stats.chisquare(obs, exp * obs.sum() / exp.sum()).pvalue > 1e-4


def test_reproducibility(gpu_ctx, models, shortlist_assets):
    m = models["tiny"]
    sents = synth.make_sentences(64, (3, 14), seed=304)
    tokens, lengths = util.pad_batch(sents)
    sp = {"temperature": 1.0, "seed": 99}
    a = m.forward(tokens, lengths, sampling=sp)
    b = m.forward(tokens, lengths, sampling=sp)
    assert np.array_equal(a["step_tokens"], b["step_tokens"])
    c = m.forward(tokens, lengths, sampling={"temperature": 1.0, "seed": 100})
    assert (c["step_tokens"] != a["step_tokens"]).any(axis=0).mean() > 0.5
    # a row of the batch equals the same sentence alone with the same key, up to the shorter step limit
    for i in (0, 17, 63):
        t1, l1 = util.pad_batch([sents[i]])
        alone = m.forward(t1, l1, sampling={"temperature": 1.0, "seed": 99, "keys": [i]})
        n = min(alone["steps"], a["steps"])
        assert np.array_equal(alone["step_tokens"][:n, 0], a["step_tokens"][:n, i]), i
    # device-resident keys equal host keys
    keys = np.arange(1000, 1064, dtype=np.uint64)[::-1].copy()
    host = m.forward(tokens, lengths, want_scores=True, sampling={"temperature": 0.7, "seed": 3, "keys": keys})
    B, T = tokens.shape
    max_steps = int(np.float32(1.5) * np.float32(T))
    d_tok, d_len, d_keys = gpu_ctx.to_device(tokens), gpu_ctx.to_device(lengths), gpu_ctx.to_device(keys)
    d_steps, d_scores = gpu_ctx.dev_alloc(4 * max_steps * B), gpu_ctx.dev_alloc(4 * max_steps * B)
    steps, _ = m.forward_resident(d_tok, d_len, B, T, d_steps, d_scores=d_scores,
                                  sampling={"temperature": 0.7, "seed": 3, "keys": d_keys})
    dev_steps = gpu_ctx.from_device(d_steps, (max_steps, B), np.uint32)[:steps]
    dev_scores = gpu_ctx.from_device(d_scores, (max_steps, B), np.float32)[:steps]
    for p in (d_tok, d_len, d_keys, d_steps, d_scores):
        gpu_ctx.dev_free(p)
    assert steps == host["steps"]
    assert np.array_equal(dev_steps, host["step_tokens"])
    assert np.array_equal(dev_scores, host["scores"])


def test_translate_independent_of_lanes_replicas_and_order(gpu_ctx, tiny_model, shortlist_assets, monkeypatch):
    sl_bin = open(shortlist_assets[0], "rb").read()
    model_bin = open(tiny_model[0], "rb").read()
    r1, r2 = capi.Model(gpu_ctx, model_bin), capi.Model(gpu_ctx, model_bin)
    sents = synth.make_sentences(60, (2, 24), seed=305)
    sp = {"temperature": 0.9, "seed": 42}
    runs = []
    for lanes, replicas in (("1", None), ("2", None), ("2", [r1, r2])):
        monkeypatch.setenv("SLIMT_B200_LANES", lanes)
        outs, st = r1.translate(sents, max_words=160, shortlist_bin=sl_bin, replicas=replicas, want_scores=True,
                                sampling=sp)
        assert st["batches"] > 2
        runs.append(([o.tolist() for o in outs], [s.tolist() for s in st["scores"]]))
    assert runs[0] == runs[1] == runs[2]
    greedy, _ = r1.translate(sents, max_words=160, shortlist_bin=sl_bin)
    assert [o.tolist() for o in greedy] != runs[0][0]
    try:  # one replica per GPU when there are two
        ctx1 = capi.Context(1)
    except RuntimeError:
        ctx1 = None
    if ctx1 is not None:
        r3 = capi.Model(ctx1, model_bin)
        outs, _ = r1.translate(sents, max_words=160, shortlist_bin=sl_bin, replicas=[r1, r3], sampling=sp)
        assert [o.tolist() for o in outs] == runs[0][0]
        r3.close()
        ctx1.close()
    # permuting the sentences with their keys permutes the output (equal lengths, no shortlist: the same batches)
    monkeypatch.delenv("SLIMT_B200_LANES")
    same = synth.make_sentences(40, (9, 9), seed=306)
    keys = np.arange(40, dtype=np.uint64) * 7919
    base, _ = r1.translate(same, max_words=90, sampling={**sp, "keys": keys})
    perm = np.random.RandomState(1).permutation(40)
    moved, _ = r1.translate([same[i] for i in perm], max_words=90, sampling={**sp, "keys": keys[perm]})
    assert [o.tolist() for o in moved] == [base[i].tolist() for i in perm]
    # the default key is the sentence's index in the request
    default, _ = r1.translate(same, max_words=90, sampling=sp)
    indexed, _ = r1.translate(same, max_words=90, sampling={**sp, "keys": np.arange(40, dtype=np.uint64)})
    assert [o.tolist() for o in default] == [o.tolist() for o in indexed]
    r1.close()
    r2.close()


@pytest.mark.parametrize("temperature", [0.0, -1.0, math.nan, math.inf, 1e4])
def test_rejected_inputs_leave_the_model_usable(models, temperature):
    m = models["tiny"]
    sents = synth.make_sentences(4, (3, 8), seed=307)
    tokens, lengths = util.pad_batch(sents)
    with pytest.raises(RuntimeError, match="temperature"):
        m.forward(tokens, lengths, sampling={"temperature": temperature})
    with pytest.raises(RuntimeError, match="temperature"):
        m.translate(sents, max_words=64, sampling={"temperature": temperature})
    forced = np.ones((int(np.float32(1.5) * np.float32(tokens.shape[1])), 4), dtype=np.uint32)
    with pytest.raises(RuntimeError, match="forced"):
        m.forward(tokens, lengths, forced=forced, sampling={"temperature": 1.0})
    # the next calls on the same model succeed: sampled, and greedy as before
    ok = m.forward(tokens, lengths, sampling={"temperature": 1.0, "seed": 1})
    assert ok["steps"] >= 1
    assert np.array_equal(m.forward(tokens, lengths)["step_tokens"], m.forward(tokens, lengths, want_logits=True)["step_tokens"])


@pytest.mark.parametrize("use_sl", [False, True], ids=["full", "shortlist"])
def test_launch_counts_equal_the_scores_route(gpu_ctx, models, shortlist_assets, use_sl):
    """sample_step takes score_step's slot: with the same number of executed steps, the same launches."""
    m = models["tiny"]
    sents = synth.make_sentences(32, (20, 20), seed=308)
    tokens, lengths = util.pad_batch(sents)
    sl = _shortlist(sents, shortlist_assets) if use_sl else None

    def run(**kw):
        gpu_ctx.profile(True)
        l0 = gpu_ctx.launches()
        m.forward(tokens, lengths, shortlist=sl, limit_factor=0.2, **kw)  # 4 steps
        n = gpu_ctx.launches() - l0
        prof = {r["name"]: r["launches"] for r in gpu_ctx.profile_read()}
        gpu_ctx.profile(False)
        return n, prof

    n_sc, p_sc = run(want_scores=True)
    for temperature in (1.0, 0.7):
        n_sa, p_sa = run(sampling={"temperature": temperature, "seed": 1})
        assert p_sa["dec_gemm_out_scores"] == p_sc["dec_gemm_out_scores"] == 4
        assert p_sa.pop("sample_step") == p_sc["score_step"] and "score_step" not in p_sa
        p_sa["score_step"] = p_sc["score_step"]
        assert p_sa == p_sc and n_sa == n_sc
