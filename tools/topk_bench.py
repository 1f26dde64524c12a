"""Cost of top-k sampling on the headline workload: tiny11 + lexical shortlist, one batch of 4096 synthetic sentences x
32 tokens, 48 decode steps at most, inputs and outputs resident on the device.  Greedy, greedy + scores, full sampling
and top-k sampling at k = 1, 10, 50 and 256 (all at temperature 1) alternate in one process (same clocks, warm L2 and
caches), in both arithmetic modes; then one profiled call of each gives the per-kernel times
(slimt_b200_profile_enable).  The card's name and power limit are read in the same process.  Prints one JSON object and
writes it to --out.
usage: python tools/topk_bench.py [--reps 10] [--out FILE]"""
import argparse
import json
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from scores_bench import LIMIT, card  # noqa: E402
from slimt_b200 import capi, synth  # noqa: E402

VARIANTS = ("greedy", "greedy_scores", "sampled", "topk_1", "topk_10", "topk_50", "topk_256")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--sentences", type=int, default=4096)
    ap.add_argument("--length", type=int, default=32)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    ctx = capi.Context(0)
    tmp = tempfile.mkdtemp(prefix="topk_bench_")
    path = os.path.join(tmp, "model.bin")
    synth.write_model(path, synth.make_params(synth.TINY, seed=1234))
    fr, offs, lists = synth.make_shortlist(vocab=32000, frequent=100, best=100, seed=7)
    sl_path = os.path.join(tmp, "lex.s2t.bin")
    synth.write_shortlist(sl_path, fr, offs, lists, best=100)
    model = capi.Model(ctx, open(path, "rb").read())
    sents = synth.make_sentences(args.sentences, args.length, seed=1000)
    B, T = len(sents), max(len(s) for s in sents)
    tok = np.zeros((B, T), dtype=np.uint32)
    lens = np.array([len(s) for s in sents], dtype=np.uint32)
    for i, s in enumerate(sents):
        tok[i, :len(s)] = s
    sl = capi.shortlist_generate(open(sl_path, "rb").read(), np.concatenate(sents), 32000)
    max_steps = max(1, int(np.float32(LIMIT) * np.float32(T)))
    d_tok, d_len, d_sl = ctx.to_device(tok), ctx.to_device(lens), ctx.to_device(sl)
    d_steps, d_scores = ctx.dev_alloc(4 * max_steps * B), ctx.dev_alloc(4 * max_steps * B)

    def call(variant):
        scores = d_scores if variant == "greedy_scores" else 0
        sampling = None
        if variant == "sampled":
            sampling = {"temperature": 1.0, "seed": 1}
        elif variant.startswith("topk"):
            sampling = {"temperature": 1.0, "seed": 1, "top_k": int(variant.split("_")[1])}
        return model.forward_resident(d_tok, d_len, B, T, d_steps, LIMIT, d_sl, len(sl), scores, sampling=sampling)

    result = {"workload": f"tiny11 + shortlist ({len(sl)} columns), {B} x {T}, {max_steps} steps at most, "
                          "device-resident, temperature 1", "card": card(), "modes": {}}
    for mode in ("exact", "fast"):
        ctx.set_math(mode == "fast")
        for v in VARIANTS:  # warm-up: module loads, workspace growth
            call(v)
        ms = {v: [] for v in VARIANTS}
        steps = {}
        for _ in range(args.reps):
            for v in VARIANTS:
                ctx.synchronize()
                ctx.timer_start()
                steps[v], _ = call(v)
                ms[v].append(ctx.timer_stop())
        prof = {}
        for v in VARIANTS:
            ctx.profile(True)
            call(v)
            prof[v] = {r["name"]: {"launches": r["launches"], "ms": r["ms"]} for r in ctx.profile_read()}
            ctx.profile(False)
        result["modes"][mode] = {
            "decode_steps": steps,
            "call_ms": ms,
            "median_ms": {v: float(np.median(ms[v])) for v in VARIANTS},
            "profile": prof,
        }
    for p in (d_tok, d_len, d_sl, d_steps, d_scores):
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
