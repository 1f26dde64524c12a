"""GPU: sentences of 257 .. 1024 tokens.  The model's length bound (slimt_b200_model_set_max_length), the long encoder
self-attention kernel (self_attention_long.cu) against the tiled kernel and the oracle, decoder cross-attention over
more than 256 keys, the translate service and replicas at the raised bound, and the C++ services with a wrap_length
above 256.  Token, encoder-output, logit and alignment checks are BIT-EXACT, except in tolerance mode."""
import os
import subprocess

import numpy as np
import pytest

import sb_testutil as util
from oracle import slimt_oracle as so
from slimt_b200 import capi, synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def long_gpu(gpu_ctx, tiny_model):
    path, items = tiny_model
    m = capi.Model(gpu_ctx, open(path, "rb").read())
    m.set_max_length(1024)
    yield m, so.Oracle(items)
    m.close()


@pytest.fixture(scope="module")
def base_gpu(gpu_ctx, tmp_path_factory):
    """Base-shaped model: emb 512, ffn 2048, 8 heads of 64."""
    path = str(tmp_path_factory.mktemp("base") / "base.bin")
    synth.write_model(path, synth.make_params(synth.ModelDims(emb=512, ffn=2048, vocab=8000), seed=5))
    m = capi.Model(gpu_ctx, open(path, "rb").read())
    m.set_max_length(1024)
    yield m, so.Oracle(synth.read_model(path))
    m.close()


def _batch(B, T, seed, vocab=32000):
    """Ragged batch: sentence 0 at full length, the last one short, the others anywhere in [1, T]."""
    sents = synth.make_sentences(B, (1, T), vocab=vocab, seed=seed)
    sents[0] = synth.make_sentences(1, T, vocab=vocab, seed=seed + 1)[0]
    if B > 1:
        sents[-1] = synth.make_sentences(1, max(1, T // 5), vocab=vocab, seed=seed + 2)[0]
    return util.pad_batch(sents)


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


def _record(steps, B, eos=0):
    """Model::decode's record() (Model.cc:127-137): each sentence's words up to and including its first EOS."""
    out = []
    for b in range(B):
        col = [int(w) for w in steps[:, b]]
        out.append(col[:col.index(eos) + 1] if eos in col else col)
    return out


def test_length_bound(gpu_ctx, tiny_model):
    m = capi.Model(gpu_ctx, open(tiny_model[0], "rb").read())
    assert m.max_length() == (256, 1024)
    tk, ln = _batch(2, 257, seed=1)
    with pytest.raises(RuntimeError, match="exceeds the supported maximum of 256"):
        m.forward(tk, ln)
    for bad in (0, 1025, -3):
        with pytest.raises(RuntimeError, match="outside"):
            m.set_max_length(bad)
        assert m.max_length() == (256, 1024)
    m.set_max_length(1024)
    assert m.max_length() == (1024, 1024)
    assert m.forward(tk, ln, limit_factor=0.01)["steps"] >= 1
    tk, ln = _batch(1, 1025, seed=2)
    with pytest.raises(RuntimeError, match="exceeds the supported maximum of 1024"):
        m.forward(tk, ln)
    m.set_max_length(100)
    tk, ln = _batch(1, 101, seed=3)
    with pytest.raises(RuntimeError, match="exceeds the supported maximum of 100"):
        m.forward(tk, ln)
    m.close()


@pytest.mark.parametrize("shape", [(2, 257), (3, 300), (2, 512), (3, 700), (1, 1024)])
def test_long_forward_matches_oracle(long_gpu, shape):
    """Tap path (encoder output, logits, alignment rows) and the fused output-GEMM + argmax path."""
    m, orc = long_gpu
    B, T = shape
    tk, ln = _batch(B, T, seed=B * 1000 + T)
    lf = 0.05
    ref = orc.forward(tk, ln, keep=True, limit_factor=lf)
    out = m.forward(tk, ln, want_encoder=True, want_logits=True, want_alignment=True, limit_factor=lf)
    _compare(out, ref, ln, T)
    fused = m.forward(tk, ln, limit_factor=lf)
    assert np.array_equal(fused["step_tokens"], ref["step_tokens"]) and fused["target_tokens"] == out["target_tokens"]


@pytest.mark.parametrize("shape", [(24, 1024), (40, 600), (64, 300)])
def test_large_long_batches_match_per_sentence_forwards(long_gpu, shape):
    """Batches too large for the oracle: without a shortlist a sentence's output does not depend on its batch, so
    sampled sentences forwarded alone (same padded width) must give the batch's bits."""
    m, _ = long_gpu
    B, T = shape
    tk, ln = _batch(B, T, seed=7 * B + T)
    lf = 0.25
    big = m.forward(tk, ln, want_encoder=True, want_alignment=True, limit_factor=lf)
    for b in sorted({0, B - 1, B // 2}):
        one = m.forward(tk[b:b + 1], ln[b:b + 1], want_encoder=True, want_alignment=True, limit_factor=lf)
        n = one["steps"]
        assert np.array_equal(one["step_tokens"][:, 0], big["step_tokens"][:n, b])
        L = int(ln[b])
        assert np.array_equal(one["encoder_out"][0, :L], big["encoder_out"][b, :L])
        assert np.array_equal(one["alignment"][:, 0, :L], big["alignment"][:n, b, :L])


@pytest.mark.parametrize("T", [257, 300, 400, 556])
def test_long_kernel_equals_tiled_tiny(long_gpu, T, monkeypatch):
    _long_vs_tiled(long_gpu[0], T, monkeypatch)


@pytest.mark.parametrize("T", [257, 300, 400])
def test_long_kernel_equals_tiled_base(base_gpu, T, monkeypatch):
    _long_vs_tiled(base_gpu[0], T, monkeypatch, vocab=8000)


def _long_vs_tiled(m, T, monkeypatch, vocab=32000):
    """Where both kernels hold the sentence, forcing either gives the same encoder output bits."""
    tk, ln = _batch(3, T, seed=31 * T, vocab=vocab)
    outs = {}
    for kern in ("tiled", "long"):
        monkeypatch.setenv("SLIMT_B200_SELFATTN", kern)
        outs[kern] = m.forward(tk, ln, want_encoder=True, limit_factor=0.02)
    monkeypatch.delenv("SLIMT_B200_SELFATTN")
    valid = np.arange(T)[None, :] < np.asarray(ln)[:, None]
    assert np.array_equal(outs["tiled"]["encoder_out"][valid], outs["long"]["encoder_out"][valid])
    assert np.array_equal(outs["tiled"]["step_tokens"], outs["long"]["step_tokens"])


def test_forced_kernels_refuse_lengths_they_cannot_hold(long_gpu, monkeypatch):
    m, _ = long_gpu
    tk, ln = _batch(2, 700, seed=5)
    for kern in ("tiled", "rowwise"):
        monkeypatch.setenv("SLIMT_B200_SELFATTN", kern)
        with pytest.raises(RuntimeError, match="sequence length 700"):
            m.forward(tk, ln, limit_factor=0.01)
    monkeypatch.delenv("SLIMT_B200_SELFATTN")
    assert m.forward(tk, ln, limit_factor=0.01)["steps"] >= 1


@pytest.mark.parametrize("T", [300, 600])
def test_base_model_long_matches_oracle(base_gpu, T):
    m, orc = base_gpu
    tk, ln = _batch(2, T, seed=T + 9, vocab=8000)
    lf = 0.03
    ref = orc.forward(tk, ln, keep=True, limit_factor=lf)
    out = m.forward(tk, ln, want_encoder=True, want_logits=True, want_alignment=True, limit_factor=lf)
    _compare(out, ref, ln, T)


def test_translate_service_long(long_gpu):
    """One request with sentences of 8 .. 1024 tokens: Batcher order, per-batch forwards, record() trimming, full
    1.5 x T decoding; and the alignments of one long sentence through the service equal the forward's tap."""
    m, _ = long_gpu
    rng = np.random.RandomState(4)
    lens = [8, 1024, 37, 300, 257, 700, 512, 999, 64, 128, 600, 1000, 16]
    sents = [synth.make_sentences(1, n, seed=int(rng.randint(1 << 30)))[0] for n in lens]
    max_words = 2048
    outs, stats = m.translate(sents, max_words=max_words)
    plan = util.batcher_generate_py(lens, max_words)
    assert stats["batches"] == len(plan)
    total = 0
    for ids, width in plan:
        tk, ln = util.pad_batch([sents[i] for i in ids])
        assert tk.shape[1] == width
        want = _record(m.forward(tk, ln)["step_tokens"], len(ids))
        for r, i in enumerate(ids):
            assert outs[i].tolist() == want[r], f"sentence {i} ({lens[i]} tokens)"
            total += len(want[r])
    assert stats["target_tokens"] == total

    s = sents[lens.index(999)]
    outs, stats = m.translate([s], max_words=max_words, want_alignments=True)
    tk, ln = util.pad_batch([s])
    fwd = m.forward(tk, ln, want_alignment=True)
    n = len(outs[0])
    assert outs[0].tolist() == _record(fwd["step_tokens"], 1)[0]
    assert np.array_equal(stats["alignments"][0], fwd["alignment"][:n, 0, :len(s)])


def test_translate_multi_applies_smallest_bound(gpu_ctx, tiny_model):
    blob = open(tiny_model[0], "rb").read()
    a, b = capi.Model(gpu_ctx, blob), capi.Model(gpu_ctx, blob)
    a.set_max_length(1024)
    sents = [synth.make_sentences(1, n, seed=n)[0] for n in (300, 12, 280)]
    with pytest.raises(RuntimeError, match="exceeds the supported maximum of 256"):
        a.translate(sents, max_words=1024, limit_factor=0.2, replicas=[a, b])
    b.set_max_length(299)
    with pytest.raises(RuntimeError, match="exceeds the supported maximum of 299"):
        b.translate(sents, max_words=1024, limit_factor=0.2, replicas=[b, a])
    b.set_max_length(512)
    multi, _ = a.translate(sents, max_words=1024, limit_factor=0.2, replicas=[a, b])
    single, _ = a.translate(sents, max_words=1024, limit_factor=0.2)
    assert [x.tolist() for x in multi] == [x.tolist() for x in single]
    a.close(), b.close()


def test_tolerance_mode_long_runs(tiny_model):
    """Tolerance mode at 700 tokens: no kernel refuses the shape.  Not bit-checked (that mode is not exact)."""
    ctx = capi.Context(0)
    ctx.set_math(True)
    m = capi.Model(ctx, open(tiny_model[0], "rb").read())
    m.set_max_length(1024)
    tk, ln = _batch(3, 700, seed=77)
    out = m.forward(tk, ln, limit_factor=0.2)
    assert out["steps"] >= 1 and (out["step_tokens"] < m.V).all()
    m.close()
    ctx.close()


def test_cpp_blocking_with_wrap_length_600(gpu_ctx, tmp_path):
    """slimt::Model admits every length the model can encode, so Blocking is bounded by wrap_length alone: a line of
    more than 256 pieces with wrap_length 600 is one segment, and its target words equal the ctypes path's."""
    spm = pytest.importorskip("sentencepiece")
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "slimt_b200", "csrc"), "host_text"])
    spm_path = os.path.join(ROOT, "tests", "golden", "text", "spm_unigram.model")
    sp = spm.SentencePieceProcessor(model_file=spm_path)
    wrap = 600
    line = " ".join(["one line long enough for a segment of more than 256 pieces, ça va?"] * 8)
    ids = sp.encode(line, out_type=int)
    assert 256 < len(ids) < wrap - 1
    text = line + "\nshort line"
    path = str(tmp_path / "m.bin")
    synth.write_model(path, synth.make_params(synth.ModelDims(vocab=sp.get_piece_size()), seed=77, eos_bias=3.0))
    binp = os.path.join(ROOT, "tests", "cpp", "host_text_test")
    r = subprocess.run([binp, path, spm_path, "-", "sentence", str(wrap), "4096", text.encode().hex()],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    lines = r.stdout.strip().split("\n")
    seg = next(l for l in lines if l.startswith("seg"))
    got_segments = [list(map(int, g.split(","))) for g in seg.split()[1:]]
    want_segments = [sp.encode(l, out_type=int) + [0] for l in text.split("\n")]
    assert got_segments == want_segments and len(got_segments[0]) > 256
    model = capi.Model(gpu_ctx, open(path, "rb").read())
    model.set_max_length(1024)
    outs, _ = model.translate([np.asarray(s, np.uint32) for s in want_segments], max_words=4096)
    src, tgt = [l for l in lines if l.startswith("blocking ")][:2]
    gaps = [bytes.fromhex(f[1:]).decode() if f != "G-" else "" for f in src.split(" ", 2)[2].split() if f.startswith("G")]
    want_text = "".join(gaps[s] + sp.decode([int(x) for x in outs[s]]) for s in range(len(outs))) + gaps[-1]
    thex = tgt.split(" ", 2)[2].split(" ", 1)[0]
    assert (bytes.fromhex(thex).decode() if thex != "-" else "") == want_text
    model.close()
