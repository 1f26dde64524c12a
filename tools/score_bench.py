"""Cost of scoring given translations on the headline workload: tiny11 + lexical shortlist, one batch of 4096 synthetic
sentences x 32 tokens, the targets being their greedy translations (EOS included).  Two ways of getting the same
numbers alternate in one process (same clocks, warm L2 and caches):
  score      slimt_b200_score, the time-parallel scoring pass, on flat host buffers (the call a user makes): host clock
             around the call, and the device time it reports
  step_path  slimt_b200_model_forward with forced = the targets and token_scores, inputs and outputs resident on the
             device (the only way to score before; it pays no host copies): CUDA events around the call
  step_path_host  the same call on host buffers (what a user of the step path pays): host clock around the call
Both are checked to give the same bits at every position the step path executed.  Then one profiled call of each gives
the per-kernel times (slimt_b200_profile_enable).  The card's name and power limit are read in the same process.
Prints one JSON object and writes it to --out.
usage: python tools/score_bench.py [--reps 10] [--out FILE]"""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from scores_bench import LIMIT, card  # noqa: E402
from slimt_b200 import capi, synth  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--sentences", type=int, default=4096)
    ap.add_argument("--length", type=int, default=32)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    ctx = capi.Context(0)
    tmp = tempfile.mkdtemp(prefix="score_bench_")
    path = os.path.join(tmp, "model.bin")
    synth.write_model(path, synth.make_params(synth.TINY, seed=1234))
    fr, offs, lists = synth.make_shortlist(vocab=32000, frequent=100, best=100, seed=7)
    sl_path = os.path.join(tmp, "lex.s2t.bin")
    synth.write_shortlist(sl_path, fr, offs, lists, best=100)
    sl_bin = open(sl_path, "rb").read()
    model = capi.Model(ctx, open(path, "rb").read())
    sents = synth.make_sentences(args.sentences, args.length, seed=1000)
    B, T = len(sents), max(len(s) for s in sents)
    max_words = B * T  # one batch, the one bench.py runs
    outs, _ = model.translate(sents, max_words=max_words, limit_factor=LIMIT, shortlist_bin=sl_bin)
    n_tgt = int(sum(len(o) for o in outs))
    Tt = max(len(o) for o in outs)

    # the step path's inputs, resident on the device
    tok = np.zeros((B, T), dtype=np.uint32)
    lens = np.array([len(s) for s in sents], dtype=np.uint32)
    for i, s in enumerate(sents):
        tok[i, :len(s)] = s
    sl = capi.shortlist_generate(sl_bin, np.concatenate(sents), 32000)
    max_steps = max(1, int(np.float32(LIMIT) * np.float32(T)))
    forced = np.zeros((max_steps, B), dtype=np.uint32)
    for b, o in enumerate(outs):
        forced[:len(o), b] = o
    d_tok, d_len, d_sl, d_forced = ctx.to_device(tok), ctx.to_device(lens), ctx.to_device(sl), ctx.to_device(forced)
    d_steps, d_scores = ctx.dev_alloc(4 * max_steps * B), ctx.dev_alloc(4 * max_steps * B)

    def step_path():
        return model.forward_resident(d_tok, d_len, B, T, d_steps, LIMIT, d_sl, len(sl), d_scores, d_forced)

    src = np.concatenate(sents).astype(np.uint32)
    src_off = np.zeros(B + 1, np.uint64)
    src_off[1:] = np.cumsum([len(x) for x in sents])
    tgt = np.concatenate(outs).astype(np.uint32)
    tgt_off = np.zeros(B + 1, np.uint64)
    tgt_off[1:] = np.cumsum([len(x) for x in outs])
    sl_buf = (capi.C.c_char * len(sl_bin)).from_buffer_copy(sl_bin)

    def score():
        flat, st = capi.score_flat([model], src, src_off, tgt, tgt_off, max_words, sl_buf)
        return [flat[int(tgt_off[b]):int(tgt_off[b + 1])] for b in range(B)], st

    def step_path_host():
        return model.forward(tok, lens, LIMIT, shortlist=sl, forced=forced, want_scores=True)

    # the same bits, at every position the step path executed
    got, st = score()
    steps, _ = step_path()
    ref = ctx.from_device(d_scores, (max_steps, B), np.float32)
    for b, o in enumerate(outs):
        n = min(len(o), steps)
        assert np.array_equal(got[b][:n].view(np.uint32), ref[:n, b].view(np.uint32)), f"sentence {b} differs"

    step_path_host()  # warm-up of the host-buffer variant
    ms = {"score": [], "step_path": [], "step_path_host": []}
    device_ms = []
    for _ in range(args.reps):
        ctx.synchronize()
        t0 = time.perf_counter()
        flat, st = capi.score_flat([model], src, src_off, tgt, tgt_off, max_words, sl_buf)
        ms["score"].append(1e3 * (time.perf_counter() - t0))
        device_ms.append(st["device_ms"])
        ctx.synchronize()
        ctx.timer_start()
        step_path()
        ms["step_path"].append(ctx.timer_stop())
        ctx.synchronize()
        t0 = time.perf_counter()
        step_path_host()
        ms["step_path_host"].append(1e3 * (time.perf_counter() - t0))
    prof = {}
    for name, fn in (("score", score), ("step_path", step_path)):
        ctx.profile(True)
        fn()
        prof[name] = {r["name"]: {"launches": r["launches"], "ms": r["ms"]} for r in ctx.profile_read()}
        ctx.profile(False)
    med = {k: float(np.median(v)) for k, v in ms.items()}
    result = {
        "workload": f"tiny11 + shortlist ({len(sl)} columns), {B} x {T} sources, their greedy translations as targets "
                    f"({n_tgt} tokens, longest {Tt})",
        "card": card(),
        "timing": "score: host clock around the C-ABI call (host buffers, shortlist generation, copies included), "
                  "score_device_ms: the CUDA-event time the call reports; step_path: CUDA events around model_forward "
                  "on device-resident buffers; step_path_host: host clock around model_forward on host buffers",
        "call_ms": ms,
        "median_ms": med,
        "score_device_ms_median": float(np.median(device_ms)),
        "target_tokens_per_s": {k: n_tgt / (med[k] / 1e3) for k in med},
        "step_path_steps": int(steps),
        "profile": prof,
    }
    for p in (d_tok, d_len, d_sl, d_forced, d_steps, d_scores):
        ctx.dev_free(p)
    model.close()
    ctx.close()
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
