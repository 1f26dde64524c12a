"""Cost of beam search on the headline workload: tiny11 + lexical shortlist, one batch of 4096 synthetic sentences x 32
tokens, 48 decode steps at most, through the translate service (host buffers in and out, as a user calls it).  Greedy
(exact arithmetic) and beam search at K = 1, 2, 4, 8 alternate in one process (same clocks, warm L2 and caches); then one
profiled call of each gives the launches and per-kernel times (slimt_b200_profile_enable).  Per variant: median ms per
call (CUDA-event time of the pass and host wall time), decoder steps executed, target tok/s of the best hypotheses and
launches per step.  The card's name and power limit are read in the same process.  Prints one JSON object and writes it
to --out.
usage: python tools/beam_bench.py [--reps 5] [--out FILE]"""
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

VARIANTS = ("greedy", "beam1", "beam2", "beam4", "beam8")
PER_STEP = ("dec_ssru_q_fused", "dec_cross_attention", "dec_cross_attention_rc", "beam_cross_attention",
            "dec_wo_ffn_fused", "dec_gemm_out_argmax", "dec_gemm_out_scores", "beam_topk", "beam_merge")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--sentences", type=int, default=4096)
    ap.add_argument("--length", type=int, default=32)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    ctx = capi.Context(0)
    ctx.set_math(False)
    tmp = tempfile.mkdtemp(prefix="beam_bench_")
    path = os.path.join(tmp, "model.bin")
    synth.write_model(path, synth.make_params(synth.TINY, seed=1234))
    fr, offs, lists = synth.make_shortlist(vocab=32000, frequent=100, best=100, seed=7)
    sl_path = os.path.join(tmp, "lex.s2t.bin")
    synth.write_shortlist(sl_path, fr, offs, lists, best=100)
    sl_bin = open(sl_path, "rb").read()
    model = capi.Model(ctx, open(path, "rb").read())
    sents = synth.make_sentences(args.sentences, args.length, seed=1000)
    max_words = len(sents) * args.length  # one batch

    def call(v):
        if v == "greedy":
            outs, st = model.translate(sents, max_words, LIMIT, sl_bin)
            st["steps"] = None
            return sum(len(o) for o in outs), st
        k = int(v[4:])
        _, st = model.translate_beam(sents, max_words, k, 1, 0.0, LIMIT, sl_bin)
        return sum(len(t) for t in st["tokens"]), st

    result = {"workload": f"tiny11 + shortlist, {len(sents)} x {args.length}, "
                          f"{max(1, int(np.float32(LIMIT) * np.float32(args.length)))} steps at most, translate service, "
                          "exact arithmetic", "card": card(), "variants": {}}
    for v in VARIANTS:  # warm-up: module loads, workspace and staging growth
        call(v)
    dev = {v: [] for v in VARIANTS}
    wall = {v: [] for v in VARIANTS}
    toks, steps = {}, {}
    for _ in range(args.reps):
        for v in VARIANTS:
            t0 = time.perf_counter()
            toks[v], st = call(v)
            wall[v].append(1e3 * (time.perf_counter() - t0))
            dev[v].append(st["device_ms"])
            steps[v] = st["steps"]
    for v in VARIANTS:
        ctx.profile(True)
        _, st = call(v)
        prof = {r["name"]: {"launches": r["launches"], "ms": r["ms"]} for r in ctx.profile_read()}
        ctx.profile(False)
        n_steps = steps[v] if steps[v] is not None else prof["dec_ssru_q_fused"]["launches"] // 2
        med = float(np.median(dev[v]))
        result["variants"][v] = {
            "median_device_ms": med,
            "median_wall_ms": float(np.median(wall[v])),
            "device_ms": dev[v],
            "steps": n_steps,
            "best_target_tokens": toks[v],
            "best_target_tok_per_s": toks[v] / (med / 1e3),
            "launches": sum(r["launches"] for r in prof.values()),
            "launches_per_step": sum(prof[t]["launches"] for t in PER_STEP if t in prof) / n_steps,
            "profile": prof,
        }
    model.close()
    ctx.close()
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
