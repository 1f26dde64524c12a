"""Launch accounting and output hashes of every decode mode, one JSON line per case.

Each line holds the case's name, a hash of every output array, and, where one context ran the whole call, its per-tag
[launches, ops, bytes] from the profiling counters.  The service cases also record kernel_launches, h2d_bytes and
d2h_bytes.  Two builds that differ only in host code must write identical files:

    python tools/launch_ab.py out_a.jsonl                              # the in-tree library
    SLIMT_B200_LIB=/path/to/other.so python tools/launch_ab.py out_b.jsonl
    cmp out_a.jsonl out_b.jsonl

Needs a B200.  Models, sentences and shortlists are generated from fixed seeds in a temporary directory.
"""
from __future__ import annotations

import hashlib
import json
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from slimt_b200 import capi, synth  # noqa: E402


def h(a):
    """Hash of the dtype, shape and bytes of an array, or of every array of a list (None stays None)."""
    if a is None:
        return None
    d = hashlib.sha256()
    for x in a if isinstance(a, list) else [a]:
        x = np.ascontiguousarray(x)
        d.update(f"{x.dtype}{x.shape}".encode())
        d.update(x.tobytes())
    return d.hexdigest()[:16]


def tags(ctx):
    return {s["name"]: [s["launches"], s["ops"], s["bytes"]] for s in sorted(ctx.profile_read(), key=lambda s: s["name"])}


def padded(sents):
    T = max(len(s) for s in sents)
    tokens = np.zeros((len(sents), T), dtype=np.uint32)
    for i, s in enumerate(sents):
        tokens[i, :len(s)] = s
    return tokens, np.array([len(s) for s in sents], dtype=np.uint32)


def sentences(n, T, seed):
    """n sentences of 3 .. T tokens, the first exactly T long."""
    out = synth.make_sentences(n, (min(3, T), T), seed=seed)
    out[0] = synth.make_sentences(1, T, seed=seed + 1)[0]
    return out


def main(path):
    tmp = tempfile.mkdtemp(prefix="slimt_b200_launch_ab_")
    ctx = capi.Context(0)
    models = {}
    for name, dims, seed in (("tiny", synth.TINY, 1234), ("base", synth.BASE, 4321)):
        mp = os.path.join(tmp, name + ".bin")
        synth.write_model(mp, synth.make_params(dims, seed=seed))
        models[name] = capi.Model(ctx, open(mp, "rb").read())
    fr, offs, lists = synth.make_shortlist(vocab=32000, frequent=100, best=100, seed=7)
    sl_path = os.path.join(tmp, "lex.bin")
    synth.write_shortlist(sl_path, fr, offs, lists, best=100)
    sl_bin = open(sl_path, "rb").read()
    lines = []

    def emit(case, out, t=None, **extra):
        rec = {"case": case, "out": out}
        rec.update(extra)
        if t is not None:
            rec["tags"] = t
        lines.append(json.dumps(rec, sort_keys=True))
        print(lines[-1][:160], flush=True)

    # ---- model_forward: every mode, both arithmetic modes, with and without a shortlist, T <= 32, 33-64, 65-256
    # (B * T above 4096 takes the recompute cross-attention, B * T below it the cached one)
    modes = ["greedy", "scores", "logits", "align", "forced", "sampled", "topk", "resident"]
    for model_name, shapes in (("tiny", ((16, 20), (96, 50), (48, 120))), ("base", ((16, 30), (64, 90)))):
        m = models[model_name]
        for B, T in shapes:
            sents = sentences(B, T, seed=B * 1000 + T)
            tokens, lengths = padded(sents)
            sl = capi.shortlist_generate(sl_bin, np.concatenate(sents), m.V)
            max_steps = max(1, int(np.float32(1.5) * np.float32(T)))
            forced = np.random.RandomState(T).randint(1, m.V, size=(max_steps, B)).astype(np.uint32)
            for math in ("exact", "fast"):
                ctx.set_math(math == "fast")
                for use_sl in (False, True):
                    for mode in modes if model_name == "tiny" else ["greedy", "scores", "align", "sampled"]:
                        Bm = 4 if mode == "logits" else B  # the logits tap of every step: a small batch
                        kw = dict(shortlist=sl if use_sl else None)
                        if mode == "scores":
                            kw["want_scores"] = True
                        elif mode == "logits":
                            kw["want_logits"] = True
                        elif mode == "align":
                            kw["want_alignment"] = True
                        elif mode == "forced":
                            kw.update(forced=forced[:, :Bm], want_scores=True)
                        elif mode == "sampled":
                            kw.update(sampling={"temperature": 0.8, "seed": 5, "keys": None}, want_scores=True)
                        elif mode == "topk":
                            kw.update(sampling={"temperature": 1.0, "seed": 3, "top_k": 10}, want_scores=True)
                        case = f"{model_name} B{Bm} T{T} {math} sl{int(use_sl)} {mode}"
                        ctx.profile(True)
                        if mode == "resident":
                            d_tok, d_len = ctx.to_device(tokens), ctx.to_device(lengths)
                            d_steps, d_sc = ctx.dev_alloc(4 * max_steps * B), ctx.dev_alloc(4 * max_steps * B)
                            d_sl = ctx.to_device(sl) if use_sl else 0
                            steps, tt = m.forward_resident(d_tok, d_len, B, T, d_steps, 1.5, d_sl, len(sl) if use_sl else 0,
                                                           d_scores=d_sc)
                            t = tags(ctx)
                            out = {"step_tokens": h(ctx.from_device(d_steps, (max_steps, B), np.uint32)[:steps]),
                                   "scores": h(ctx.from_device(d_sc, (max_steps, B), np.float32)[:steps]),
                                   "steps": steps, "target_tokens": tt}
                            for p in (d_tok, d_len, d_steps, d_sc, d_sl):
                                if p:
                                    ctx.dev_free(p)
                        else:
                            r = m.forward(tokens[:Bm], lengths[:Bm], **kw)
                            t = tags(ctx)
                            out = {k: h(r[k]) for k in ("step_tokens", "scores", "logits", "alignment")}
                            out.update(steps=r["steps"], target_tokens=r["target_tokens"])
                        ctx.profile(False)
                        emit(case, out, t)
    ctx.set_math(False)

    # ---- the service entry points
    def service(case, fn, lanes, **extra):
        os.environ["SLIMT_B200_LANES"] = str(lanes)
        ctx.profile(True)
        out, st = fn()
        t = tags(ctx) if lanes == 1 else None  # with two lanes, which batches lane 0 served depends on timing
        ctx.profile(False)
        for k in ("kernel_launches", "h2d_bytes", "d2h_bytes", "batches"):
            out[k] = st[k]
        emit(case, out, t, lanes=lanes, **extra)

    tiny = models["tiny"]
    req = synth.make_sentences(300, (3, 40), seed=77)

    def translate(sl, align, scores, sampling=None, replicas=None):
        def run():
            outs, st = tiny.translate(req, max_words=1024, shortlist_bin=sl_bin if sl else None, replicas=replicas,
                                      want_alignments=align, want_scores=scores, sampling=sampling)
            return {"tokens": h(outs), "scores": h(st.get("scores")), "alignments": h(st.get("alignments")),
                    "target_tokens": st["target_tokens"]}, st
        return run

    for math in ("exact", "fast"):
        ctx.set_math(math == "fast")
        for lanes in (1, 2):
            for sl in (False, True):
                service(f"translate_multi {math} lanes{lanes} sl{int(sl)} align scores",
                        translate(sl, True, True, replicas=[tiny]), lanes)
            service(f"translate_sampled {math} lanes{lanes} sl1 scores",
                    translate(True, False, True, {"temperature": 0.7, "seed": 11, "keys": np.arange(300)[::-1] * 3}),
                    lanes)
            service(f"translate_topk {math} lanes{lanes} sl1 scores",
                    translate(True, False, True, {"temperature": 1.0, "seed": 2, "top_k": 5}), lanes)
    ctx.set_math(False)

    def beam(K, nbest, sl, align, sents=req):
        def run():
            nb, st = tiny.translate_beam(sents, max_words=1024, beam_size=K, nbest=nbest, length_penalty=0.6,
                                         shortlist_bin=sl_bin if sl else None, want_alignments=align)
            flat = [x for hyps in nb for x in hyps]
            return {"nbest_tokens": h([x["tokens"] for x in flat]), "nbest_scores": h([x["scores"] for x in flat]),
                    "nbest_totals": h(np.array([x["total"] for x in flat], np.float32)),
                    "nbest_normalized": h(np.array([x["normalized"] for x in flat], np.float64)),
                    "tokens": h(st["tokens"]), "scores": h(st["scores"]), "alignments": h(st.get("alignments")),
                    "steps": st["steps"], "target_tokens": st["target_tokens"]}, st
        return run

    for K in (1, 4, 8):
        for sl in (False, True):
            for align in (False, True):
                service(f"translate_beam K{K} nbest{K} sl{int(sl)} align{int(align)}", beam(K, K, sl, align), 1)
    for lanes in (1, 2):
        service(f"translate_beam K4 nbest2 sl1 align1 lanes{lanes}", beam(4, 2, True, True), lanes)
    # K = 1 is greedy decoding bit for bit: tokens, scores and alignments of the best hypothesis
    os.environ["SLIMT_B200_LANES"] = "1"
    for sl in (False, True):
        g, gs = tiny.translate(req, max_words=1024, shortlist_bin=sl_bin if sl else None, want_alignments=True,
                               want_scores=True)
        _, bs = tiny.translate_beam(req, max_words=1024, beam_size=1, shortlist_bin=sl_bin if sl else None,
                                    want_alignments=True)
        same = (all(np.array_equal(x, y) for x, y in zip(g, bs["tokens"])) and
                all(np.array_equal(x, y) for x, y in zip(gs["scores"], bs["scores"])) and
                all(np.array_equal(x, y) for x, y in zip(gs["alignments"], bs["alignments"])))
        emit(f"translate_beam K1 equals greedy sl{int(sl)}", {"equal": bool(same), "tokens": h(g)})

    def score(srcs, tgts, sl, align, max_words):
        def run():
            sc, st = tiny.score(srcs, tgts, max_words=max_words, shortlist_bin=sl_bin if sl else None,
                                want_alignments=align)
            return {"scores": h(sc), "alignments": h(st.get("alignments"))}, st
        return run

    tgts = synth.make_sentences(300, (1, 60), seed=78)
    for lanes in (1, 2):
        for sl in (False, True):
            for align in (False, True):
                service(f"score lanes{lanes} sl{int(sl)} align{int(align)}", score(req, tgts, sl, align, 1024), lanes)
    # one batch of 400 x 48 = 19 200 rows: the output layer in two chunks
    big_src = synth.make_sentences(400, 10, seed=79)
    big_tgt = synth.make_sentences(400, 48, seed=80)
    for align in (False, True):
        service(f"score one batch 19200 rows sl1 align{int(align)}", score(big_src, big_tgt, True, align, 8192), 1)
    os.environ.pop("SLIMT_B200_LANES")

    with open(path, "w") as f:
        f.write("\n".join(lines) + "\n")
    print(f"{len(lines)} cases -> {path}")


if __name__ == "__main__":
    main(sys.argv[1])
