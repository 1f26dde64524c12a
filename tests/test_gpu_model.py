"""GPU: Model::forward through the C ABI against the oracle and the reference-generated golden vectors.
Everything is compared BIT-EXACT (tokens, encoder output, logits, alignment probabilities)."""
import numpy as np
import pytest

import golden_cases
import sb_testutil as util
from oracle import slimt_oracle as so
from slimt_b200 import capi, synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def tiny_gpu(gpu_ctx, tiny_model):
    path, items = tiny_model
    m = capi.Model(gpu_ctx, open(path, "rb").read())
    yield m, so.Oracle(items)
    m.close()


@pytest.fixture(scope="module")
def eos_gpu(gpu_ctx, eos_model):
    path, items = eos_model
    m = capi.Model(gpu_ctx, open(path, "rb").read())
    yield m, so.Oracle(items)
    m.close()


def _compare(out, ref, lengths, T):
    valid = np.arange(T)[None, :] < np.asarray(lengths)[:, None]
    assert out["steps"] == len(ref["step_tokens"])
    assert np.array_equal(out["step_tokens"], ref["step_tokens"])
    assert out["target_tokens"] == sum(len(s) for s in ref["sentences"])
    if out["encoder_out"] is not None:
        assert np.array_equal(out["encoder_out"][valid], ref["encoder_out"][valid])
    if out["logits"] is not None:
        for s in range(out["steps"]):
            assert np.array_equal(out["logits"][s], ref["logits"][s]), f"logits differ at step {s}"
    if out["alignment"] is not None:
        a = np.stack([x[:, 0, 0, :] for x in ref["attn"]])
        assert np.array_equal(out["alignment"][:, valid], a[:, valid])


@pytest.mark.parametrize("name", sorted(golden_cases.FORWARD_CASES))
def test_golden_forward(gpu_ctx, name, tmp_path):
    path, tokens, lengths, sl, forced, g = golden_cases.load_case(name, tmp_path)
    m = capi.Model(gpu_ctx, open(path, "rb").read())
    out = m.forward(tokens, lengths, shortlist=sl, forced=forced, want_encoder=True, want_logits=True, want_alignment=True)
    golden_cases.check_against_golden(g, lengths, out["step_tokens"], out["encoder_out"], out["logits"], out["alignment"])
    fused = m.forward(tokens, lengths, shortlist=sl, forced=forced)  # fused output-GEMM + argmax path
    assert np.array_equal(fused["step_tokens"], g["step_tokens"])
    m.close()


@pytest.mark.parametrize("shape", [(8, 16), (5, 9), (1, 1), (3, 33), (130, 7), (6, 64), (3, 100), (2, 256)])
def test_forward_ragged_batches(tiny_gpu, shape):
    """Includes the long end of BASELINE.json's mixed-length sweep (8-256 tokens): keys beyond one 32-row box,
    the cached K/V cross-attention path and hundreds of decode steps."""
    m, orc = tiny_gpu
    B, T = shape
    sents = synth.make_sentences(B, (1, T), seed=B * 100 + T)
    sents[0] = synth.make_sentences(1, T, seed=1)[0]
    tokens, lengths = util.pad_batch(sents)
    ref = orc.forward(tokens, lengths, keep=True)
    out = m.forward(tokens, lengths, want_encoder=True, want_logits=True, want_alignment=True)
    _compare(out, ref, lengths, T)
    fused = m.forward(tokens, lengths)
    assert np.array_equal(fused["step_tokens"], ref["step_tokens"]) and fused["target_tokens"] == out["target_tokens"]


@pytest.mark.parametrize("shape", [(37, 32), (9, 20), (4, 32), (5, 33), (7, 64), (41, 48), (3, 40), (130, 64), (2, 57)])
def test_cross_attention_recompute_equals_cached_path(tiny_gpu, shape, monkeypatch):
    """S <= 32 batches re-project K/V on the tensor cores every step (cross_attention_rc.cu); forcing the cached
    f32 K/V kernel must give the same bits, and both must equal the oracle."""
    m, orc = tiny_gpu
    B, T = shape
    sents = synth.make_sentences(B, (1, T), seed=7 * B + T)
    sents[0] = synth.make_sentences(1, T, seed=2)[0]
    sents[-1] = synth.make_sentences(1, T, seed=3)[0]
    tokens, lengths = util.pad_batch(sents)
    ref = orc.forward(tokens, lengths, keep=True)
    monkeypatch.setenv("SLIMT_B200_CROSS", "rc")  # (small batches would take the cached kernel by themselves)
    rc = m.forward(tokens, lengths, want_logits=True, want_alignment=True)
    monkeypatch.setenv("SLIMT_B200_CROSS", "cached")
    cached = m.forward(tokens, lengths, want_logits=True, want_alignment=True)
    monkeypatch.delenv("SLIMT_B200_CROSS")
    _compare(rc, ref, lengths, T)
    _compare(cached, ref, lengths, T)
    assert np.array_equal(rc["logits"], cached["logits"])


@pytest.mark.parametrize("shape", [(5, 65), (3, 100), (4, 128), (3, 129), (2, 256), (150, 70), (6, 200), (9, 255)])
def test_long_sentence_cross_attention_recompute_equals_cached_path(tiny_gpu, shape, monkeypatch):
    """Batches of 65 .. 256 source tokens re-project K/V a sentence at a time (cross_attention_rcl_kernel in
    cross_attention_rc.cu: one or two 128-key groups per sentence, softmax across the groups, one weighted-sum chain
    carried over them; ragged lengths from 1 token up, more sentences than SMs).  Forcing the cached f32 K/V kernel
    must give the same bits, and both must equal the oracle."""
    m, orc = tiny_gpu
    B, T = shape
    sents = synth.make_sentences(B, (1, T), seed=17 * B + T)
    sents[0] = synth.make_sentences(1, T, seed=2)[0]
    sents[-1] = synth.make_sentences(1, max(1, T - 3), seed=3)[0]
    tokens, lengths = util.pad_batch(sents)
    lf = 0.25 if B * T <= 1024 else 0.1
    monkeypatch.setenv("SLIMT_B200_CROSS", "rc")
    rc = m.forward(tokens, lengths, want_logits=True, want_alignment=True, limit_factor=lf)
    monkeypatch.setenv("SLIMT_B200_CROSS", "cached")
    cached = m.forward(tokens, lengths, want_logits=True, want_alignment=True, limit_factor=lf)
    monkeypatch.delenv("SLIMT_B200_CROSS")
    assert np.array_equal(rc["logits"], cached["logits"])
    assert np.array_equal(rc["alignment"], cached["alignment"])
    assert np.array_equal(rc["step_tokens"], cached["step_tokens"])
    if B * T <= 1024:  # the oracle's share of the check, at sizes it finishes in seconds
        ref = orc.forward(tokens, lengths, keep=True, limit_factor=lf)
        _compare(rc, ref, lengths, T)


@pytest.mark.parametrize("shape", [(37, 32), (9, 20), (70, 5), (130, 1), (5, 33), (7, 64), (40, 48), (3, 2)])
def test_fused_encoder_attention_equals_split_path(tiny_gpu, shape, monkeypatch):
    """T <= 64 batches run the q/k/v projections and the self-attention as one kernel (enc_attention.cu): tiles of
    floor(128 / T) whole sentences, sentences straddling warps, ragged lengths.  Forcing the split path (three GEMMs
    writing f32 Q, K, V + self_attention_kernel) must give the same bits, and both must equal the oracle."""
    m, orc = tiny_gpu
    B, T = shape
    sents = synth.make_sentences(B, (1, T), seed=11 * B + T)
    sents[0] = synth.make_sentences(1, T, seed=2)[0]
    sents[-1] = synth.make_sentences(1, T, seed=3)[0]
    tokens, lengths = util.pad_batch(sents)
    ref = orc.forward(tokens, lengths, keep=True)
    fused = m.forward(tokens, lengths, want_encoder=True, want_logits=True)
    monkeypatch.setenv("SLIMT_B200_SELFATTN", "split")
    split = m.forward(tokens, lengths, want_encoder=True, want_logits=True)
    monkeypatch.delenv("SLIMT_B200_SELFATTN")
    _compare(split, ref, lengths, T)
    _compare(fused, ref, lengths, T)
    valid = np.arange(T)[None, :] < np.asarray(lengths)[:, None]
    assert np.array_equal(fused["encoder_out"][valid], split["encoder_out"][valid])
    assert np.array_equal(fused["logits"], split["logits"])


@pytest.mark.parametrize("shape", [(5, 70), (3, 129), (2, 256), (9, 33), (40, 8), (3, 200)])
def test_tiled_self_attention_equals_rowwise_kernel(tiny_gpu, shape, monkeypatch):
    """The split path's attention kernel exists twice: the register-tiled one (self_attention_tiled.cu: 64 query rows
    per block, partial key tiles, sentences straddling query blocks) and the first one-thread-per-query kernel.  Same
    chains, so the same bits -- and both equal the oracle."""
    m, orc = tiny_gpu
    B, T = shape
    sents = synth.make_sentences(B, (1, T), seed=13 * B + T)
    sents[0] = synth.make_sentences(1, T, seed=2)[0]
    sents[-1] = synth.make_sentences(1, max(1, T - 1), seed=3)[0]
    tokens, lengths = util.pad_batch(sents)
    monkeypatch.setenv("SLIMT_B200_SELFATTN", "tiled")
    tiled = m.forward(tokens, lengths, want_encoder=True)
    monkeypatch.setenv("SLIMT_B200_SELFATTN", "rowwise")
    rowwise = m.forward(tokens, lengths, want_encoder=True)
    monkeypatch.delenv("SLIMT_B200_SELFATTN")
    valid = np.arange(T)[None, :] < np.asarray(lengths)[:, None]
    assert np.array_equal(tiled["encoder_out"][valid], rowwise["encoder_out"][valid])
    assert np.array_equal(tiled["step_tokens"], rowwise["step_tokens"])
    ref = orc.forward(tokens, lengths, keep=True)
    assert np.array_equal(tiled["encoder_out"][valid], ref["encoder_out"][valid])


def test_forward_with_shortlist(tiny_gpu, shortlist_assets):
    m, orc = tiny_gpu
    fr, offs, lists = shortlist_assets[1]
    sents = synth.make_sentences(12, (3, 14), seed=8)
    tokens, lengths = util.pad_batch(sents)
    sl = so.shortlist_generate(np.concatenate(sents), fr, offs, lists, 32000)
    ref = orc.forward(tokens, lengths, shortlist=sl, keep=True)
    out = m.forward(tokens, lengths, shortlist=sl, want_logits=True)
    _compare(out, ref, lengths, tokens.shape[1])
    assert np.isin(out["step_tokens"], sl).all()
    assert np.array_equal(m.forward(tokens, lengths, shortlist=sl)["step_tokens"], ref["step_tokens"])


def test_eos_bookkeeping_and_early_stop(eos_gpu):
    m, orc = eos_gpu
    sents = synth.make_sentences(8, (4, 10), seed=33)
    tokens, lengths = util.pad_batch(sents)
    ref = orc.forward(tokens, lengths)
    out = m.forward(tokens, lengths)
    assert len({len(s) for s in ref["sentences"]}) > 1
    _compare(out, ref, lengths, tokens.shape[1])
    # a batch in which every sentence finishes early stops before the limit, like Model.cc:161
    quick = [i for i, s in enumerate(ref["sentences"]) if s[-1] == 0]
    if quick:
        tk, ln = util.pad_batch([sents[i] for i in quick])
        r2 = orc.forward(tk, ln)
        o2 = m.forward(tk, ln)
        assert o2["steps"] == len(r2["step_tokens"]) < int(1.5 * tk.shape[1]) or o2["steps"] == len(r2["step_tokens"])
        assert np.array_equal(o2["step_tokens"], r2["step_tokens"])


def test_teacher_forced_logits(tiny_gpu):
    m, orc = tiny_gpu
    sents = synth.make_sentences(6, 11, seed=2)
    tokens, lengths = util.pad_batch(sents)
    forced = np.random.RandomState(3).randint(1, 32000, size=(16, 6)).astype(np.uint32)
    ref = orc.forward(tokens, lengths, forced=forced, keep=True)
    out = m.forward(tokens, lengths, forced=forced, want_logits=True)
    _compare(out, ref, lengths, 11)


def test_batch_composition_independence_at_full_size(tiny_gpu):
    """Size-independent property at the BASELINE batch size: without a shortlist a sentence's output does not
    depend on which batch it is in, so 4096 x 32 in one batch must equal the same sentences in 64-sentence
    batches; a seeded sample of those is checked against the oracle."""
    m, orc = tiny_gpu
    sents = synth.make_sentences(4096, 32, seed=1000)
    tokens, lengths = util.pad_batch(sents)
    big = m.forward(tokens, lengths)
    assert big["steps"] == 48
    rng = np.random.RandomState(0)
    for start in rng.choice(64, size=3, replace=False) * 64:
        small = m.forward(tokens[start:start + 64], lengths[start:start + 64])
        n = small["steps"]
        assert np.array_equal(small["step_tokens"], big["step_tokens"][:n, start:start + 64])
    ref = orc.forward(tokens[:16], lengths[:16])
    assert np.array_equal(big["step_tokens"][:, :16], ref["step_tokens"])


def test_translate_service_matches_per_batch_oracle(tiny_gpu, shortlist_assets):
    """slimt_b200_translate == exhaust(): Batcher order, per-batch shortlist union, record() trimming."""
    m, orc = tiny_gpu
    sl_path, (fr, offs, lists) = shortlist_assets
    sents = synth.make_sentences(40, (2, 12), seed=77)
    outs, stats = m.translate(sents, max_words=96, shortlist_bin=open(sl_path, "rb").read())
    plan = util.batcher_generate_py([len(s) for s in sents], 96)
    assert stats["batches"] == len(plan)
    total = 0
    for ids, width in plan:
        chunk = [sents[i] for i in ids]
        tk, ln = util.pad_batch(chunk)
        assert tk.shape[1] == width
        sl = so.shortlist_generate(np.concatenate(chunk), fr, offs, lists, 32000)
        ref = orc.forward(tk, ln, shortlist=sl)
        for r, i in enumerate(ids):
            assert outs[i].tolist() == ref["sentences"][r], f"sentence {i}"
            total += len(ref["sentences"][r])
    assert stats["target_tokens"] == total
    assert stats["kernel_launches"] > 0 and stats["h2d_bytes"] > 0 and stats["d2h_bytes"] > 0


def test_base_shaped_model(gpu_ctx, tmp_path):
    """BASELINE configs[2]: emb 512, ffn 2048 (head size 64)."""
    path = str(tmp_path / "base.bin")
    dims = synth.ModelDims(emb=512, ffn=2048, vocab=8000)
    synth.write_model(path, synth.make_params(dims, seed=5))
    m = capi.Model(gpu_ctx, open(path, "rb").read())
    orc = so.Oracle(synth.read_model(path))
    sents = synth.make_sentences(6, (2, 10), vocab=8000, seed=6)
    tokens, lengths = util.pad_batch(sents)
    ref = orc.forward(tokens, lengths, keep=True)
    out = m.forward(tokens, lengths, want_encoder=True, want_logits=True)
    _compare(out, ref, lengths, tokens.shape[1])
    m.close()


def test_error_paths(gpu_ctx, tiny_model):
    path, _ = tiny_model
    blob = bytearray(open(path, "rb").read())
    blob[0] = 9
    with pytest.raises(RuntimeError, match="versions do not match"):
        capi.Model(gpu_ctx, bytes(blob))
    m = capi.Model(gpu_ctx, open(path, "rb").read())
    with pytest.raises(RuntimeError, match="multiple of 8"):
        m.forward(np.ones((2, 4), np.uint32), np.array([4, 4], np.uint32), shortlist=np.arange(5, dtype=np.uint32))
    out = m.forward(np.zeros((0, 4), np.uint32), np.zeros(0, np.uint32))
    assert out["steps"] == 0 and out["target_tokens"] == 0
    m.close()


def test_malformed_model_images_are_reported_not_followed(gpu_ctx, tiny_model):
    """io::load_items trusts nothing in the header here: counts, name / shape tables and blob sizes are checked against
    what is left of the image (a truncated or garbage file is an error, as the reference's MmapFile / ABORT_IF paths)."""
    import struct
    path, _ = tiny_model
    good = open(path, "rb").read()
    for cut in (8, 24, 16 + 32 * 10, 16 + 32 * 193 + 100, 16 + 32 * 193 + 5000, len(good) // 2, len(good) - 300):
        with pytest.raises(RuntimeError, match="truncated|too small|missing|unexpected|not a 2-D"):
            capi.Model(gpu_ctx, good[:cut])
    huge = bytearray(good)
    struct.pack_into("<Q", huge, 8, 1 << 60)  # item count
    with pytest.raises(RuntimeError, match="truncated"):
        capi.Model(gpu_ctx, bytes(huge))
    names = bytearray(good)
    struct.pack_into("<Q", names, 16, 1 << 40)  # first item's name length
    with pytest.raises(RuntimeError, match="truncated"):
        capi.Model(gpu_ctx, bytes(names))
    shape = bytearray(good)
    struct.pack_into("<Q", shape, 16 + 16, 1 << 20)  # first item's rank
    with pytest.raises(RuntimeError, match="truncated or malformed"):
        capi.Model(gpu_ctx, bytes(shape))


def test_translate_rejects_bad_requests_before_any_gpu_work(tiny_gpu, shortlist_assets):
    m, _ = tiny_gpu
    ok = synth.make_sentences(4, (3, 9), seed=1)
    launches = m.ctx.launches()
    with pytest.raises(RuntimeError, match="exceeds the supported maximum"):
        m.translate(ok + [np.ones(300, np.uint32)], max_words=4096)
    with pytest.raises(RuntimeError, match="empty sentences"):
        m.translate(ok + [np.zeros(0, np.uint32)], max_words=4096)
    assert m.ctx.launches() == launches, "a request that cannot be served must fail as a whole, before any batch runs"
    bad_sl = bytearray(open(shortlist_assets[0], "rb").read())
    bad_sl[-2] = 0xFF  # a target id far beyond the vocabulary
    with pytest.raises(RuntimeError, match="out of bounds"):
        m.translate([np.array([31999, 0], np.uint32)], max_words=64, shortlist_bin=bytes(bad_sl))
