"""Cost of per-token scores on the headline workload: tiny11 + lexical shortlist, one batch of 4096 synthetic sentences
x 32 tokens, inputs and outputs resident on the device.  Calls with and without scores alternate in one process (same
clocks, warm L2 and caches), in both arithmetic modes; then one profiled call of each gives the per-kernel times
(slimt_b200_profile_enable) of the fused argmax GEMM against the scores GEMM and the step kernel.  Prints one JSON object
and writes it to --out.  usage: python tools/scores_bench.py [--reps 10] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from slimt_b200 import capi, synth  # noqa: E402

LIMIT = 1.5


def card():
    """Name and power limit of device 0, read in the same process as the measurement."""
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [x.strip() for x in q.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clock}
    except Exception as e:  # noqa: BLE001 -- reported, not hidden
        return {"name": None, "error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--sentences", type=int, default=4096)
    ap.add_argument("--length", type=int, default=32)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    ctx = capi.Context(0)
    tmp = tempfile.mkdtemp(prefix="scores_bench_")
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

    def call(scores):
        return model.forward_resident(d_tok, d_len, B, T, d_steps, LIMIT, d_sl, len(sl), d_scores if scores else 0)

    result = {"workload": f"tiny11 + shortlist ({len(sl)} columns), {B} x {T}, device-resident", "card": card(),
              "modes": {}}
    for mode in ("exact", "fast"):
        ctx.set_math(mode == "fast")
        for scores in (False, True):  # warm-up: module loads, workspace growth
            call(scores)
        ms = {False: [], True: []}
        for _ in range(args.reps):
            for scores in (False, True):
                ctx.synchronize()
                ctx.timer_start()
                steps, _ = call(scores)
                ms[scores].append(ctx.timer_stop())
        tokens_off = ctx.from_device(d_steps, (max_steps, B), np.uint32)[:steps].copy()
        call(True)
        tokens_on = ctx.from_device(d_steps, (max_steps, B), np.uint32)[:steps]
        sc = ctx.from_device(d_scores, (max_steps, B), np.float32)[:steps]
        prof = {}
        for scores in (False, True):
            ctx.profile(True)
            call(scores)
            prof["on" if scores else "off"] = {r["name"]: {"launches": r["launches"], "ms": r["ms"]}
                                               for r in ctx.profile_read()}
            ctx.profile(False)
        result["modes"][mode] = {
            "decode_steps": steps,
            "call_ms_off": ms[False], "call_ms_on": ms[True],
            "median_ms_off": float(np.median(ms[False])), "median_ms_on": float(np.median(ms[True])),
            "tokens_equal": bool(np.array_equal(tokens_off, tokens_on)),
            "score_range": [float(sc.min()), float(sc.max())],
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
