"""GPU: top-k sampling (include/slimt_b200.h, DESIGN §4.4e).  Each step's word is drawn from S_k, the first min(k, N)
columns by (logit descending, column ascending), with the CDF over S_k in ascending column order; the reference below
recomputes u in numpy and that CDF in float64 from the logits tap of the same call."""
import ctypes as C

import numpy as np
import pytest
from scipy import stats

import sb_testutil as util
from oracle import slimt_oracle as so
from slimt_b200 import capi, synth
from test_gpu_large_golden import _periodic_model
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


def _uniform(seed, keys, step):
    B = len(keys)
    return uniform_np(np.full(B, seed, dtype=np.uint64), keys, np.full(B, step, dtype=np.uint64)).astype(np.float64) * 2.0**-53


def _sets(y, k):
    """S_k of every row of y [B][N], in ascending column order: [B][min(k, N)]."""
    N = y.shape[1]
    order = np.lexsort((np.broadcast_to(np.arange(N), y.shape), -y), axis=-1)
    return np.sort(order[:, :min(k, N)], axis=1)


def _check_topk(out, temperature, seed, keys, sl, k):
    """Every row of every executed step of a call made with want_logits and want_scores.  Returns the number of draws
    whose u was clear of every CDF boundary (compared exactly)."""
    inv_t = _inv_t(temperature)
    B = out["step_tokens"].shape[1]
    keys = np.arange(B, dtype=np.uint64) if keys is None else np.asarray(keys, dtype=np.uint64)
    exact = 0
    for s in range(out["steps"]):
        y = out["logits"][s]
        sk = _sets(y, k)
        words = out["step_tokens"][s].astype(np.int64)
        cols = words if sl is None else np.searchsorted(sl, words)
        if sl is not None:
            assert np.array_equal(sl[cols], words)
        r = np.arange(B)
        assert (sk == cols[:, None]).any(axis=1).all(), f"step {s}: a word outside S_k"
        i = np.argmax(sk == cols[:, None], axis=1)
        z = (y[r[:, None], sk] * inv_t).astype(np.float32).astype(np.float64)
        M = z.max(axis=1)
        p = np.exp(z - M[:, None])
        S = p.sum(axis=1)
        F = np.cumsum(p, axis=1) / S[:, None]
        u = _uniform(seed, keys, s)
        lo = np.where(i > 0, F[r, np.maximum(i - 1, 0)], 0.0)
        assert (lo - EPS <= u).all() and (u <= F[r, i] + EPS).all(), s
        clear = np.abs(F - u[:, None]).min(axis=1) > EPS
        want = np.array([np.searchsorted(F[b], u[b], side="right") for b in range(B)])
        assert np.array_equal(i[clear], want[clear]), s
        exact += int(clear.sum())
        sc = out["scores"][s].astype(np.float64)
        assert np.isfinite(sc).all()
        assert np.abs(sc - (z[r, i] - (M + np.log(S)))).max() <= TOL, s
    return exact


# ---------------------------------------------------------------- every row of every step, and the two routes
@pytest.mark.parametrize("k", [1, 2, 10, 256])
@pytest.mark.parametrize("temperature", [0.5, 1.0, 2.0])
@pytest.mark.parametrize("use_sl", [False, True], ids=["full", "shortlist"])
@pytest.mark.parametrize("which", ["tiny", "eos"])
def test_against_float64_and_routes(models, shortlist_assets, which, use_sl, temperature, k):
    m = models[which]
    sents = synth.make_sentences(24, (2, 16), seed=401)
    tokens, lengths = util.pad_batch(sents)
    sl = _shortlist(sents, shortlist_assets) if use_sl else None
    sp = {"temperature": temperature, "seed": 11, "top_k": k}
    tap = m.forward(tokens, lengths, shortlist=sl, want_logits=True, want_scores=True, sampling=sp)
    assert _check_topk(tap, temperature, 11, None, sl, k) > 0
    bare = m.forward(tokens, lengths, shortlist=sl, want_scores=True, sampling=sp)
    assert bare["steps"] == tap["steps"]
    assert np.array_equal(bare["step_tokens"], tap["step_tokens"])
    assert np.array_equal(bare["scores"], tap["scores"])


@pytest.mark.parametrize("use_sl", [False, True], ids=["full", "shortlist"])
def test_tolerance_mode_against_its_tap(fast_model, shortlist_assets, use_sl):
    sents = synth.make_sentences(16, (3, 16), seed=402)
    tokens, lengths = util.pad_batch(sents)
    sl = _shortlist(sents, shortlist_assets) if use_sl else None
    sp = {"temperature": 0.8, "seed": 5, "keys": np.arange(100, 116, dtype=np.uint64), "top_k": 10}
    tap = fast_model.forward(tokens, lengths, shortlist=sl, want_logits=True, want_scores=True, sampling=sp)
    assert _check_topk(tap, 0.8, 5, sp["keys"], sl, 10) > 0
    bare = fast_model.forward(tokens, lengths, shortlist=sl, want_scores=True, sampling=sp)
    assert np.array_equal(bare["step_tokens"], tap["step_tokens"]) and np.array_equal(bare["scores"], tap["scores"])


# ---------------------------------------------------------------- k = 1 is greedy; k >= N is unrestricted
@pytest.mark.parametrize("use_sl", [False, True], ids=["full", "shortlist"])
@pytest.mark.parametrize("which", ["tiny", "eos"])
def test_k1_is_greedy(models, shortlist_assets, which, use_sl):
    m = models[which]
    sents = synth.make_sentences(40, (2, 20), seed=403)
    tokens, lengths = util.pad_batch(sents)
    sl = _shortlist(sents, shortlist_assets) if use_sl else None
    greedy = m.forward(tokens, lengths, shortlist=sl)
    for temperature, seed in ((1.0, 0), (0.3, 7), (2.5, 2**63 + 5)):
        out = m.forward(tokens, lengths, shortlist=sl, want_scores=True,
                        sampling={"temperature": temperature, "seed": seed, "top_k": 1})
        assert out["steps"] == greedy["steps"]
        assert np.array_equal(out["step_tokens"], greedy["step_tokens"])
        assert (out["scores"] == 0.0).all()


def test_k_at_least_n_follows_the_unrestricted_draw(models):
    m = models["tiny"]
    sents = synth.make_sentences(64, (4, 16), seed=404)
    tokens, lengths = util.pad_batch(sents)
    sl = np.sort(np.random.RandomState(5).choice(32000, 128, replace=False)).astype(np.uint32)
    sl[0] = 0  # EOS
    sl = np.sort(sl)
    keys = np.arange(500, 564, dtype=np.uint64)
    sp = {"temperature": 1.0, "seed": 21, "keys": keys}
    topk = m.forward(tokens, lengths, shortlist=sl, want_logits=True, sampling={**sp, "top_k": 256})
    full = m.forward(tokens, lengths, shortlist=sl, sampling=sp)
    B, compared = tokens.shape[0], 0
    same_so_far = np.ones(B, dtype=bool)
    for s in range(min(topk["steps"], full["steps"])):
        z = topk["logits"][s].astype(np.float64)
        p = np.exp(z - z.max(axis=1, keepdims=True))
        F = np.cumsum(p, axis=1) / p.sum(axis=1, keepdims=True)
        u = _uniform(21, keys, s)
        clear = np.abs(F - u[:, None]).min(axis=1) > EPS
        check = same_so_far & clear
        assert np.array_equal(topk["step_tokens"][s][check], full["step_tokens"][s][check]), s
        compared += int(check.sum())
        same_so_far &= topk["step_tokens"][s] == full["step_tokens"][s]
    assert compared >= B


# ---------------------------------------------------------------- ties, distribution
@pytest.mark.parametrize("period", [256, 1000])
def test_ties_take_the_lowest_columns(gpu_ctx, tmp_path, period):
    path = str(tmp_path / f"periodic_{period}.bin")
    _periodic_model(path, period)
    m = capi.Model(gpu_ctx, open(path, "rb").read())
    sents = synth.make_sentences(32, (3, 12), seed=405)
    tokens, lengths = util.pad_batch(sents)
    out = m.forward(tokens, lengths, want_logits=True, want_scores=True,
                    sampling={"temperature": 1.0, "seed": 8, "top_k": 10})
    assert _check_topk(out, 1.0, 8, None, None, 10) > 0
    # the ties are real: S_10's columns hold fewer than 10 distinct values somewhere
    y0 = out["logits"][0]
    sk = _sets(y0, 10)
    assert min(len(np.unique(y0[b, sk[b]])) for b in range(len(sents))) < 10
    m.close()


def test_distribution_chi_square(models):
    m = models["tiny"]
    sent = synth.make_sentences(1, (8, 8), seed=406)[0]
    one_t, one_l = util.pad_batch([sent])
    y = m.forward(one_t, one_l, want_logits=True)["logits"][0]
    sk = _sets(y, 10)[0]
    z = y[0, sk].astype(np.float64)
    p = np.exp(z - z.max())
    p /= p.sum()
    B = 4096
    tokens, lengths = np.tile(one_t, (B, 1)), np.tile(one_l, B)
    out = m.forward(tokens, lengths, limit_factor=0.01, sampling={"temperature": 1.0, "seed": 2025, "top_k": 10})
    words = out["step_tokens"][0].astype(np.int64)
    assert np.isin(words, sk).all(), "a word outside S_10"
    counts = np.array([(words == c).sum() for c in sk])
    expected = B * p
    big = expected >= 5
    obs, exp = counts[big], expected[big]
    if (~big).any():
        obs, exp = np.append(obs, counts[~big].sum()), np.append(exp, expected[~big].sum())
    assert big.sum() >= 2
    assert stats.chisquare(obs, exp * obs.sum() / exp.sum()).pvalue > 1e-4


# ---------------------------------------------------------------- reproducibility
def test_reproducibility(gpu_ctx, models):
    m = models["tiny"]
    sents = synth.make_sentences(64, (3, 14), seed=407)
    tokens, lengths = util.pad_batch(sents)
    sp = {"temperature": 1.0, "seed": 99, "top_k": 50}
    a = m.forward(tokens, lengths, sampling=sp)
    b = m.forward(tokens, lengths, sampling=sp)
    assert np.array_equal(a["step_tokens"], b["step_tokens"])
    c = m.forward(tokens, lengths, sampling={**sp, "seed": 100})
    assert (c["step_tokens"] != a["step_tokens"]).any(axis=0).mean() > 0.5
    for i in (0, 17, 63):
        t1, l1 = util.pad_batch([sents[i]])
        alone = m.forward(t1, l1, sampling={**sp, "keys": [i]})
        n = min(alone["steps"], a["steps"])
        assert np.array_equal(alone["step_tokens"][:n, 0], a["step_tokens"][:n, i]), i
    keys = np.arange(1000, 1064, dtype=np.uint64)[::-1].copy()
    sk = {"temperature": 0.7, "seed": 3, "top_k": 10}
    host = m.forward(tokens, lengths, want_scores=True, sampling={**sk, "keys": keys})
    B, T = tokens.shape
    max_steps = int(np.float32(1.5) * np.float32(T))
    d_tok, d_len, d_keys = gpu_ctx.to_device(tokens), gpu_ctx.to_device(lengths), gpu_ctx.to_device(keys)
    d_steps, d_scores = gpu_ctx.dev_alloc(4 * max_steps * B), gpu_ctx.dev_alloc(4 * max_steps * B)
    steps, _ = m.forward_resident(d_tok, d_len, B, T, d_steps, d_scores=d_scores, sampling={**sk, "keys": d_keys})
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
    sents = synth.make_sentences(60, (2, 24), seed=408)
    sp = {"temperature": 0.9, "seed": 42, "top_k": 10}
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
    monkeypatch.delenv("SLIMT_B200_LANES")
    same = synth.make_sentences(40, (9, 9), seed=409)
    keys = np.arange(40, dtype=np.uint64) * 7919
    base, _ = r1.translate(same, max_words=90, sampling={**sp, "keys": keys})
    perm = np.random.RandomState(2).permutation(40)
    moved, _ = r1.translate([same[i] for i in perm], max_words=90, sampling={**sp, "keys": keys[perm]})
    assert [o.tolist() for o in moved] == [base[i].tolist() for i in perm]
    default, _ = r1.translate(same, max_words=90, sampling=sp)
    indexed, _ = r1.translate(same, max_words=90, sampling={**sp, "keys": np.arange(40, dtype=np.uint64)})
    assert [o.tolist() for o in default] == [o.tolist() for o in indexed]
    r1.close()
    r2.close()


def test_top_k_zero_is_the_sampled_call(models, shortlist_assets):
    m = models["eos"]
    sents = synth.make_sentences(32, (2, 16), seed=410)
    tokens, lengths = util.pad_batch(sents)
    sl = _shortlist(sents, shortlist_assets)
    sp = {"temperature": 0.8, "seed": 6}
    a = m.forward(tokens, lengths, shortlist=sl, want_scores=True, sampling=sp)
    b = m.forward(tokens, lengths, shortlist=sl, want_scores=True, sampling={**sp, "top_k": 0})
    assert a["steps"] == b["steps"]
    assert np.array_equal(a["step_tokens"], b["step_tokens"]) and np.array_equal(a["scores"], b["scores"])
    sl_bin = open(shortlist_assets[0], "rb").read()
    ta, sa = m.translate(sents, max_words=128, shortlist_bin=sl_bin, want_scores=True, sampling=sp)
    tb, sb = m.translate(sents, max_words=128, shortlist_bin=sl_bin, want_scores=True, sampling={**sp, "top_k": 0})
    assert [o.tolist() for o in ta] == [o.tolist() for o in tb]
    assert all(np.array_equal(x, y) for x, y in zip(sa["scores"], sb["scores"]))


# ---------------------------------------------------------------- rejected inputs, launches
def test_rejected_inputs_leave_the_model_usable(models):
    m = models["tiny"]
    sents = synth.make_sentences(4, (3, 8), seed=411)
    tokens, lengths = util.pad_batch(sents)
    for k in (-1, 257, 1 << 20):
        with pytest.raises(RuntimeError, match="top_k"):
            m.forward(tokens, lengths, sampling={"temperature": 1.0, "top_k": k})
        with pytest.raises(RuntimeError, match="top_k"):
            m.translate(sents, max_words=64, sampling={"temperature": 1.0, "top_k": k})
    with pytest.raises(RuntimeError, match="temperature"):
        m.forward(tokens, lengths, sampling={"temperature": 0.0, "top_k": 5})
    forced = np.ones((int(np.float32(1.5) * np.float32(tokens.shape[1])), 4), dtype=np.uint32)
    with pytest.raises(RuntimeError, match="forced"):
        m.forward(tokens, lengths, forced=forced, sampling={"temperature": 1.0, "top_k": 5})
    # top_k > 0 without sampling parameters, straight through the C ABI
    steps = np.zeros((int(np.float32(1.5) * np.float32(tokens.shape[1])), 4), dtype=np.uint32)
    io = capi.ForwardIO(tokens.ctypes.data, lengths.ctypes.data, 4, tokens.shape[1], 1.5, None, 0, None, 0,
                        steps.ctypes.data, 0, 0, None, None, None, None)
    assert capi.lib().slimt_b200_model_forward_topk(m.h, C.byref(io), None, 5) != 0
    assert b"sampling" in capi.lib().slimt_b200_last_error()
    ok = m.forward(tokens, lengths, sampling={"temperature": 1.0, "seed": 1, "top_k": 3})
    assert ok["steps"] >= 1
    assert np.array_equal(m.forward(tokens, lengths)["step_tokens"], m.forward(tokens, lengths, want_logits=True)["step_tokens"])


@pytest.mark.parametrize("use_sl", [False, True], ids=["full", "shortlist"])
def test_launch_counts_do_not_depend_on_k(gpu_ctx, models, shortlist_assets, use_sl):
    """A top-k step launches 3 * Ld + 2 kernels (DESIGN §4.4e): the sampled step's, with the logits GEMM in place of the
    scores GEMM and topk_sample in place of sample_step."""
    m = models["tiny"]
    sents = synth.make_sentences(32, (20, 20), seed=412)
    tokens, lengths = util.pad_batch(sents)
    sl = _shortlist(sents, shortlist_assets) if use_sl else None

    def run(**kw):
        gpu_ctx.profile(True)
        l0 = gpu_ctx.launches()
        out = m.forward(tokens, lengths, shortlist=sl, limit_factor=0.2, **kw)  # 4 steps
        n = gpu_ctx.launches() - l0
        prof = {r["name"]: r["launches"] for r in gpu_ctx.profile_read()}
        gpu_ctx.profile(False)
        assert out["steps"] == 4
        return n, prof

    step_tags = ("dec_ssru_q_fused", "dec_cross_attention", "dec_cross_attention_rc", "dec_wo_ffn_fused",
                 "dec_gemm_out_logits", "topk_sample")
    n_sa, p_sa = run(sampling={"temperature": 1.0, "seed": 1})
    per_step = set()
    for k in (1, 10, 256):
        n_k, p_k = run(sampling={"temperature": 1.0, "seed": 1, "top_k": k})
        per_step.add(sum(v for t, v in p_k.items() if t in step_tags) / 4)
        assert p_k.pop("topk_sample") == 4 and p_k.pop("dec_gemm_out_logits") == 4
        assert "sample_step" not in p_k and "dec_gemm_out_scores" not in p_k and "argmax_rows" not in p_k
        p_k["sample_step"], p_k["dec_gemm_out_scores"] = p_sa["sample_step"], p_sa["dec_gemm_out_scores"]
        assert p_k == p_sa and n_k == n_sa
    assert per_step == {3 * 2 + 2}
