"""GPU: the forward pass through every reachable combination of its kernel routes.  The workspace holds only the
buffers the chosen routes read, so a route that lost one of its buffers would read a null or short one: each
combination of self-attention kernel (SLIMT_B200_SELFATTN), cross-attention kernel (SLIMT_B200_CROSS and the batch
shape), encoder FFN (tiny: row-tile kernel, base: gemm_i8), output route (the fused argmax on the digits, the fused
argmax on the bound filter with the models of test_gpu_out_fallback.py at K = 256 and 512, logits tap), shortlist on
and off, host and device I/O runs in both arithmetic modes.
Exact mode must give the oracle's tokens."""
import numpy as np
import pytest

import sb_testutil as util
from oracle import slimt_oracle as so
from slimt_b200 import capi, synth
from test_gpu_out_fallback import fallback_base_model, fallback_model  # noqa: F401  (fixtures)

pytestmark = pytest.mark.gpu

# short: T <= 64, the fused encoder attention by default, SLIMT_B200_CROSS=rc takes the recompute kernel;
# long: 65 <= T <= 256, the tiled kernel by default, rc takes the sentence-at-a-time kernel in exact mode
SHAPES = {"short": (9, 40), "long": (5, 90)}
SELF = [None, "rowwise", "tiled", "long"]  # None: the default route
CROSS = ["cached", "rc"]
_oracle_cache = {}


@pytest.fixture(scope="module")
def models(gpu_ctx, tiny_model, fallback_model, fallback_base_model, tmp_path_factory):  # noqa: F811
    base_path = str(tmp_path_factory.mktemp("model") / "base.bin")
    synth.write_model(base_path, synth.make_params(synth.BASE, seed=77))
    out = {}
    for name, path in (("tiny", tiny_model[0]), ("fallback", fallback_model[0]), ("base", base_path),
                       ("fallback_base", fallback_base_model[0])):
        out[name] = (capi.Model(gpu_ctx, open(path, "rb").read()), so.Oracle(synth.read_model(path)))
    yield out
    for m, _ in out.values():
        m.close()


def _batch(shape, shortlist_assets):
    B, T = SHAPES[shape]
    sents = synth.make_sentences(B, (1, T), seed=B * 100 + T)
    sents[0] = synth.make_sentences(1, T, seed=1)[0]
    tokens, lengths = util.pad_batch(sents)
    fr, offs, lists = shortlist_assets[1]
    sl = so.shortlist_generate(np.concatenate(sents), fr, offs, lists, 32000)
    return tokens, lengths, sl


def _oracle(name, orc, shape, tokens, lengths, sl):
    key = (name, shape, sl is not None)
    if key not in _oracle_cache:
        _oracle_cache[key] = np.asarray(orc.forward(tokens, lengths, shortlist=sl)["step_tokens"])
    return _oracle_cache[key]


def _device_forward(ctx, m, tokens, lengths, sl):
    B, T = tokens.shape
    max_steps = max(1, int(np.float32(1.5) * np.float32(T)))
    ptrs = [ctx.to_device(tokens), ctx.to_device(lengths), ctx.dev_alloc(4 * max_steps * B)]
    if sl is not None:
        ptrs.append(ctx.to_device(np.ascontiguousarray(sl, dtype=np.uint32)))
    try:
        n, _ = m.forward_resident(ptrs[0], ptrs[1], B, T, ptrs[2], d_shortlist=ptrs[3] if sl is not None else 0,
                                  n_shortlist=0 if sl is None else len(sl))
        return ctx.from_device(ptrs[2], (max_steps, B), np.uint32)[:n]
    finally:
        for p in ptrs:
            ctx.dev_free(p)


@pytest.mark.parametrize("cross", CROSS)
@pytest.mark.parametrize("selfattn", SELF)
@pytest.mark.parametrize("name,shape", [("tiny", "short"), ("tiny", "long"), ("fallback", "short"),
                                        ("fallback", "long"), ("base", "short"), ("fallback_base", "short")])
def test_route_combination(gpu_ctx, models, shortlist_assets, monkeypatch, name, shape, selfattn, cross):
    m, orc = models[name]
    tokens, lengths, sl_words = _batch(shape, shortlist_assets)
    if selfattn:
        monkeypatch.setenv("SLIMT_B200_SELFATTN", selfattn)
    monkeypatch.setenv("SLIMT_B200_CROSS", cross)
    try:
        for fast in (False, True):
            gpu_ctx.set_math(fast)
            for sl in (None, sl_words):
                what = f"{'fast' if fast else 'exact'} shortlist={sl is not None}"
                if not fast:
                    # greedy decoding: the oracle's tokens, through the fused argmax and through the logits tap
                    ref = _oracle(name, orc, shape, tokens, lengths, sl)
                    for logits in (False, True):
                        out = m.forward(tokens, lengths, shortlist=sl, want_logits=logits)
                        assert np.array_equal(out["step_tokens"], ref), f"{what} logits={logits}"
                    host = out["step_tokens"]
                else:
                    # teacher forcing keeps the histories equal: the fused argmax agrees with the argmax of the same
                    # mode's float logits except at near-ties (the bar of test_gpu_fast_mode.py)
                    steps = int(np.float32(1.5) * np.float32(tokens.shape[1]))
                    forced = np.random.RandomState(3).randint(1, 32000, size=(steps, len(lengths))).astype(np.uint32)
                    tap = m.forward(tokens, lengths, shortlist=sl, forced=forced, want_logits=True)["step_tokens"]
                    fused = m.forward(tokens, lengths, shortlist=sl, forced=forced)["step_tokens"]
                    n = min(len(tap), len(fused))  # a near-tie at EOS may end the batch a step apart
                    agree = (fused[:n] == tap[:n]).mean()
                    assert agree >= 0.99, f"{what}: {agree}"
                    host = m.forward(tokens, lengths, shortlist=sl)["step_tokens"]
                # device-resident input and output: the same tokens as the host-buffer call of the same mode
                assert np.array_equal(_device_forward(gpu_ctx, m, tokens, lengths, sl), host), f"{what} device_io"
    finally:
        gpu_ctx.set_math(False)
