"""GPU: beam search (slimt_b200_translate_beam, DESIGN §4.4d).

K = 1 against greedy decoding bit for bit; K = 2, 4, 8 against a numpy beam search over the oracle's exact logits, and
against slimt_b200_score of every returned hypothesis bit for bit; independence from batch, order, replicas and lanes;
rejected inputs; the launches per step; and the headline batch at K = 4."""

import numpy as np
import pytest

import sb_testutil as util
from oracle import slimt_oracle as so
from slimt_b200 import capi, synth

pytestmark = pytest.mark.gpu
BIG = 1 << 20  # max_words large enough for one batch
LIMIT = 1.5
NEAR = 1e-4  # nats: a reference decision this close is not compared
NO_EOS_BIAS = -30.0  # the output bias on EOS that keeps every hypothesis running to the step limit


def _model(ctx, tmp_path_factory, dims, seed, eos_bias):
    path = str(tmp_path_factory.mktemp("model") / "model.bin")
    params = synth.make_params(dims, seed=seed, eos_bias=eos_bias)
    synth.write_model(path, params)
    return capi.Model(ctx, open(path, "rb").read()), synth.read_model(path)


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
def no_eos(gpu_ctx, tmp_path_factory):
    m, items = _model(gpu_ctx, tmp_path_factory, synth.TINY, 1234, NO_EOS_BIAS)
    yield m, items
    m.close()


@pytest.fixture(scope="module")
def quick_eos(gpu_ctx, tmp_path_factory):
    """An EOS bias strong enough that every sentence's K hypotheses finish within a few steps."""
    m, items = _model(gpu_ctx, tmp_path_factory, synth.TINY, 4321, 8.0)
    yield m, items
    m.close()


@pytest.fixture(scope="module")
def base(gpu_ctx, tmp_path_factory):
    m, items = _model(gpu_ctx, tmp_path_factory, synth.BASE, 77, 2.0)
    yield m, items
    m.close()


@pytest.fixture(autouse=True)
def _exact(gpu_ctx):
    gpu_ctx.set_math(False)
    yield
    gpu_ctx.set_math(False)


def _sl_bin(shortlist_assets, use_sl):
    return open(shortlist_assets[0], "rb").read() if use_sl else None


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


# ---------------------------------------------------------------- 1. K = 1 is greedy
K1_CASES = [("tiny", False, (3, 32)), ("tiny", True, (3, 32)), ("eos", False, (3, 32)), ("eos", True, (3, 32)),
            ("eos", True, (33, 64)), ("tiny", False, (65, 256)), ("eos", True, (257, 300)), ("base", True, (3, 32)),
            ("base", False, (33, 64))]


@pytest.mark.parametrize("which,use_sl,lengths", K1_CASES, ids=[f"{w}-{'sl' if s else 'full'}-{a}-{b}"
                                                                 for w, s, (a, b) in K1_CASES])
def test_k1_is_greedy(request, shortlist_assets, which, use_sl, lengths):
    m, _ = request.getfixturevalue(which)
    if lengths[1] > m.max_length()[0]:
        m.set_max_length(lengths[1])
    sents = synth.make_sentences(6, lengths, seed=11 + lengths[0])
    sl = _sl_bin(shortlist_assets, use_sl)
    want, wst = m.translate(sents, BIG, LIMIT, sl, want_alignments=True, want_scores=True)
    got, st = m.translate_beam(sents, BIG, 1, 1, 0.0, LIMIT, sl, want_alignments=True)
    for i in range(len(sents)):
        assert np.array_equal(st["tokens"][i], want[i]), f"tokens {i}"
        assert np.array_equal(got[i][0]["tokens"], want[i])
        assert np.array_equal(_bits(st["scores"][i]), _bits(wst["scores"][i])), f"scores {i}"
        assert np.array_equal(_bits(got[i][0]["scores"]), _bits(wst["scores"][i]))
        assert np.array_equal(_bits(st["alignments"][i]), _bits(wst["alignments"][i])), f"alignments {i}"


def test_k1_is_greedy_recompute_cross_attention(tiny, shortlist_assets):
    """One batch of B * T > 4096: greedy runs the recompute cross-attention, beam search the cached multi-query kernel."""
    m, _ = tiny
    sents = synth.make_sentences(160, 30, seed=5)
    sl = _sl_bin(shortlist_assets, True)
    want, wst = m.translate(sents, BIG, LIMIT, sl, want_alignments=True, want_scores=True)
    got, st = m.translate_beam(sents, BIG, 1, 1, 0.0, LIMIT, sl, want_alignments=True)
    assert st["batches"] == 1
    for i in range(len(sents)):
        assert np.array_equal(st["tokens"][i], want[i]), f"tokens {i}"
        assert np.array_equal(_bits(st["scores"][i]), _bits(wst["scores"][i])), f"scores {i}"
        assert np.array_equal(_bits(st["alignments"][i]), _bits(wst["alignments"][i])), f"alignments {i}"


# ---------------------------------------------------------------- 2. against a reference search
def _reference_search(items, sources, K, shortlist):
    """The definition of include/slimt_b200.h over Oracle.step with a float64 LSE.  Returns, per sentence, its K
    finished hypotheses in finishing order as (tokens, total f32), and whether a merge cut was within NEAR."""
    orc = so.Oracle(items)
    tokens, lengths = util.pad_batch(sources)
    B, T = tokens.shape
    mask01 = (np.arange(T)[None, :] < np.asarray(lengths)[:, None]).astype(np.float32)
    mask = ((np.float32(1) - mask01) * np.float32(-99999999.0)).astype(np.float32)
    enc = np.repeat(orc.encode(tokens, mask), K, axis=0)
    maskK = np.repeat(mask, K, axis=0)
    max_steps = max(1, int(np.float32(LIMIT) * np.float32(T)))
    states = [np.zeros((B * K, 1, orc.W.E), dtype=np.float32) for _ in range(orc.Ld)]
    width = [K] * B
    hyps = [[([], np.float32(0))] for _ in range(B)]  # live slots: (tokens, cum)
    fin = [[] for _ in range(B)]
    near = [False] * B
    prev = None
    for s in range(max_steps):
        if not any(width):
            break
        logits, _, _ = orc.step(enc, maskK, states, prev, shortlist)
        L = logits.reshape(B * K, -1).astype(np.float64)
        m = L.max(axis=1)
        lse = m + np.log(np.exp(L - m[:, None]).sum(axis=1))
        cols_all = np.arange(L.shape[1])
        nxt_prev = np.zeros(B * K, dtype=np.uint32)
        gather = np.arange(B * K)
        new_hyps = [[] for _ in range(B)]
        for b in range(B):
            w = width[b]
            if w == 0:
                continue
            cands = []
            for k, (toks, cum) in enumerate(hyps[b]):
                row = b * K + k
                y = logits.reshape(B * K, -1)[row]
                order = np.lexsort((cols_all, -y))[:K]
                for j, c in enumerate(order):
                    sc = np.float32(float(y[c]) - lse[row])
                    cands.append((np.float32(cum + sc), k, j, int(c), sc))
            cands.sort(key=lambda t: (-float(t[0]), t[1], t[2]))
            if len(cands) > w and abs(float(cands[w - 1][0]) - float(cands[w][0])) < NEAR:
                near[b] = True
            for t, k, j, c, sc in cands[:w]:
                word = int(shortlist[c]) if shortlist is not None else c
                toks = hyps[b][k][0] + [word]
                if word == 0 or s == max_steps - 1:
                    fin[b].append((toks, t))
                else:
                    n = len(new_hyps[b])
                    new_hyps[b].append((toks, t))
                    gather[b * K + n] = b * K + k
                    nxt_prev[b * K + n] = word
            width[b] = len(new_hyps[b])
        states = [st[gather] for st in states]
        hyps = new_hyps
        prev = nxt_prev
    return fin, near


def _rank(fin, alpha):
    """(tokens, total, normalized) best first; ties keep the finishing order; and whether two ranks were within NEAR."""
    ranked = sorted(((t, tot, float(tot) / (len(t) ** alpha)) for t, tot in fin), key=lambda h: -h[2])
    close = any(abs(ranked[i][2] - ranked[i + 1][2]) < NEAR for i in range(len(ranked) - 1))
    return ranked, close


_REF = {}


@pytest.mark.parametrize("K", [2, 4, 8])
@pytest.mark.parametrize("alpha", [0.0, 1.0])
@pytest.mark.parametrize("use_sl", [False, True], ids=["full", "shortlist"])
@pytest.mark.parametrize("which", ["eos", "no_eos"])
def test_matches_reference_search(request, shortlist_assets, which, use_sl, alpha, K):
    m, items = request.getfixturevalue(which)
    sents = synth.make_sentences(6, (3, 7), seed=21)
    sl = so.shortlist_generate(np.concatenate(sents), *shortlist_assets[1], 32000) if use_sl else None
    key = (which, use_sl, K)
    if key not in _REF:
        _REF[key] = _reference_search(items, sents, K, sl)
    fin, near = _REF[key]
    got, _ = m.translate_beam(sents, BIG, K, K, alpha, LIMIT, _sl_bin(shortlist_assets, use_sl))
    compared = 0
    for b in range(len(sents)):
        assert len(fin[b]) == K
        ranked, close = _rank(fin[b], alpha)
        if near[b] or close:
            continue
        compared += 1
        for h in range(K):
            assert got[b][h]["tokens"].tolist() == ranked[h][0], f"sentence {b} hypothesis {h}"
            if which == "no_eos":
                assert len(ranked[h][0]) == max(1, int(np.float32(LIMIT) * np.float32(max(len(s) for s in sents))))
    print(f"reference search {which} {'shortlist' if use_sl else 'full'} K={K} alpha={alpha}: "
          f"{compared} of {len(sents)} sentences compared")
    assert compared >= len(sents) // 2 + 1, f"only {compared} of {len(sents)} sentences free of near-ties"


# ---------------------------------------------------------------- 3. against scoring
def _check_against_scoring(m, sents, K, sl, alpha=1.0):
    got, st = m.translate_beam(sents, BIG, K, K, alpha, LIMIT, sl, want_alignments=True)
    limit = {}
    for bi_ids, width in capi.batcher_plan([len(s) for s in sents], BIG):
        for i in bi_ids:
            limit[int(i)] = max(1, int(np.float32(LIMIT) * np.float32(width)))
    for h in range(K):
        targets = [got[i][h]["tokens"] for i in range(len(sents))]
        sc, sst = m.score(sents, targets, BIG, sl, want_alignments=(h == 0))
        for i in range(len(sents)):
            hyp = got[i][h]
            assert np.array_equal(_bits(sc[i]), _bits(hyp["scores"])), f"sentence {i} hypothesis {h}"
            total = np.float32(0)
            for v in hyp["scores"]:
                total = np.float32(total + v)
            assert _bits(total) == _bits(hyp["total"])
            assert hyp["normalized"] == float(hyp["total"]) / (len(hyp["tokens"]) ** alpha)
            assert hyp["tokens"][-1] == 0 or len(hyp["tokens"]) == limit[i]
            if h == 0:
                assert np.array_equal(hyp["tokens"], st["tokens"][i])
                assert np.array_equal(_bits(sst["alignments"][i]), _bits(st["alignments"][i])), f"alignment {i}"
    for i in range(len(sents)):
        norms = [got[i][h]["normalized"] for h in range(K)]
        assert all(norms[h] >= norms[h + 1] for h in range(K - 1))
        assert len({tuple(got[i][h]["tokens"].tolist()) for h in range(K)}) == K


@pytest.mark.parametrize("K", [2, 4, 8])
@pytest.mark.parametrize("use_sl", [False, True], ids=["full", "shortlist"])
def test_matches_scoring(eos, shortlist_assets, use_sl, K):
    m, _ = eos
    sents = synth.make_sentences(24, (3, 40), seed=31)
    _check_against_scoring(m, sents, K, _sl_bin(shortlist_assets, use_sl))


# ---------------------------------------------------------------- 4. independence
def _lists(got, i):
    return [(h["tokens"].tolist(), _bits(h["scores"]).tolist(), _bits(h["total"]).tolist()) for h in got[i]]


def test_independent_of_batch_order_replicas_lanes(eos, gpu_ctx, tmp_path_factory, eos_model, monkeypatch):
    m, _ = eos
    sents = synth.make_sentences(12, 9, seed=41)  # one width, so every case has the same step limit
    K = 4
    alone = [m.translate_beam([s], BIG, K, K, 1.0)[0][0] for s in sents[:3]]
    batch, _ = m.translate_beam(sents, BIG, K, K, 1.0)
    perm = np.random.default_rng(1).permutation(len(sents))
    permuted, _ = m.translate_beam([sents[i] for i in perm], BIG, K, K, 1.0)
    m2 = capi.Model(gpu_ctx, open(eos_model[0], "rb").read())
    try:
        reps, rst = m.translate_beam(sents, 40, K, K, 1.0, replicas=[m, m2])
    finally:
        m2.close()
    assert rst["batches"] > 2
    monkeypatch.setenv("SLIMT_B200_LANES", "2")
    lanes, _ = m.translate_beam(sents, 40, K, K, 1.0)
    for i in range(3):
        assert _lists([alone[i]], 0) == _lists(batch, i)
    for j, i in enumerate(perm):
        assert _lists(permuted, j) == _lists(batch, i)
    for i in range(len(sents)):
        assert _lists(reps, i) == _lists(batch, i)
        assert _lists(lanes, i) == _lists(batch, i)


# ---------------------------------------------------------------- 5. errors
@pytest.mark.parametrize("K,nbest,alpha,cap", [(0, 1, 0.0, None), (9, 1, 0.0, None), (4, 0, 0.0, None),
                                               (4, 5, 0.0, None), (4, 2, -1.0, None), (4, 2, float("nan"), None),
                                               (4, 2, float("inf"), None), (4, 2, 0.5, 3)])
def test_rejected_inputs(eos, gpu_ctx, eos_model, K, nbest, alpha, cap):
    m, _ = eos
    sents = synth.make_sentences(5, (3, 9), seed=51)
    launches = gpu_ctx.launches()
    with pytest.raises(RuntimeError, match="beam"):
        m.translate_beam(sents, BIG, K, nbest, alpha, nbest_capacity=cap)
    assert gpu_ctx.launches() == launches, "an input error is reported before any GPU work"
    got, _ = m.translate_beam(sents, BIG, 4, 2, 0.5)
    fresh = capi.Model(gpu_ctx, open(eos_model[0], "rb").read())
    try:
        want, _ = fresh.translate_beam(sents, BIG, 4, 2, 0.5)
    finally:
        fresh.close()
    for i in range(len(sents)):
        assert _lists(got, i) == _lists(want, i)


# ---------------------------------------------------------------- 6. launches
STEP_TAGS = {"dec_ssru_q_fused": 2, "beam_cross_attention": 2, "dec_wo_ffn_fused": 2, "dec_gemm_out_scores": 1,
             "beam_topk": 1, "beam_merge": 1}


def _profiled(ctx, m, sents, K, sl):
    ctx.profile(True)
    try:
        _, st = m.translate_beam(sents, BIG, K, 1, 0.0, LIMIT, sl)
        prof = {r["name"]: r["launches"] for r in ctx.profile_read()}
    finally:
        ctx.profile(False)
    return st, prof


def test_launches_per_step(quick_eos, gpu_ctx, shortlist_assets):
    m, _ = quick_eos
    sl = _sl_bin(shortlist_assets, True)
    per_step, fixed = set(), []
    for n, K in ((8, 2), (8, 8), (40, 2), (40, 8)):
        sents = synth.make_sentences(n, 12, seed=61)
        st, prof = _profiled(gpu_ctx, m, sents, K, sl)
        assert st["batches"] == 1
        max_steps = int(np.float32(LIMIT) * np.float32(12))
        assert st["steps"] < max_steps, "the loop stops once every sentence is done"
        for tag, k in STEP_TAGS.items():
            assert prof[tag] == k * st["steps"], tag
        per_step.add(sum(prof[t] for t in STEP_TAGS) // st["steps"])
        fixed.append({t: v for t, v in prof.items() if t not in STEP_TAGS})
    assert len(per_step) == 1
    assert all(f == fixed[0] for f in fixed)


# ---------------------------------------------------------------- 7. at size
def test_headline_batch_k4(tiny, shortlist_assets):
    m, _ = tiny
    sents = synth.make_sentences(4096, 32, seed=1000)
    sl = _sl_bin(shortlist_assets, True)
    got, st = m.translate_beam(sents, 1 << 17, 4, 4, 1.0, LIMIT, sl)
    assert st["batches"] == 1
    assert all(len(got[i]) == 4 for i in range(len(sents)))
    pick = np.random.default_rng(7).choice(len(sents), size=64, replace=False)
    # scored inside the whole request, so that the batch and its shortlist union are the beam search's
    for h in range(4):
        targets = [got[i][h]["tokens"] for i in range(len(sents))]
        sc, _ = m.score(sents, targets, 1 << 17, sl)
        for i in pick:
            assert np.array_equal(_bits(sc[i]), _bits(got[i][h]["scores"])), f"sentence {i} hypothesis {h}"
