"""Long-sentence throughput of the tiny model in exact mode: 131 072 source tokens per pass as 512 x 256, 256 x 512 and
128 x 1024 full-length sentences, limit factor 1.5, inputs resident in HBM, L2 overwritten before every timed pass.

Per shape: target tokens per second over the timed passes (CUDA events), per-kernel times of one profiled pass
(slimt_b200_profile_*), and the encoder self-attention kernel's fp32 FMA rate (FMAs computed from shapes) against the
card's fp32 FMA peak (148 SMs x 128 FMA per clock x clocks.max.sm).  Then the tiled-vs-long self-attention A/B at
T in {288, 384, 448, 512} (tiny, head size 32) and {288, 384} (base, head size 64), which sets the dispatch boundary
in engine.cu.  The card's name, power limit and maximum SM
clock are read in the same run.

    python tools/long_bench.py [--reps 5] [--out FILE]
"""
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
TOKENS = 131072
SHAPES = [(512, 256), (256, 512), (128, 1024)]
AB_T = [288, 384, 448, 512]
AB_T_BASE = [288, 384]  # head size 64: the tiled kernel holds up to 400 tokens
ENC_LAYERS, HEADS = 6, 8


def card():
    q = "name,power.limit,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", "0"],
                       capture_output=True, text=True, check=True)
    name, power, mhz = [x.strip() for x in r.stdout.strip().split("\n")[0].split(",")]
    return {"gpu": name, "power_limit_w": float(power), "sm_max_mhz": float(mhz)}


class Batch:
    def __init__(self, ctx, B, T, seed, limit=LIMIT, vocab=32000):
        sents = synth.make_sentences(B, T, vocab=vocab, seed=seed)
        tok = np.stack(sents).astype(np.uint32)
        self.B, self.T, self.limit = B, T, limit
        self.max_steps = max(1, int(np.float32(limit) * np.float32(T)))
        self.tok = ctx.to_device(tok)
        self.lens = ctx.to_device(np.full(B, T, np.uint32))
        self.steps = ctx.dev_alloc(4 * self.max_steps * B)

    def run(self, model):
        return model.forward_resident(self.tok, self.lens, self.B, self.T, self.steps, self.limit)

    def free(self, ctx):
        for p in (self.tok, self.lens, self.steps):
            ctx.dev_free(p)


def profiled(ctx, model, batch):
    ctx.profile(True)
    batch.run(model)
    stats = ctx.profile_read()
    ctx.profile(False)
    return {s["name"]: {"launches": s["launches"], "ms": round(s["ms"], 4)} for s in stats}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--ab-reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    hw = card()
    peak_fma = 148 * 128 * hw["sm_max_mhz"] * 1e6
    peak_name = f"148 SMs x 128 fp32 FMA/clock x {hw['sm_max_mhz']:.0f} MHz (clocks.max.sm) = {peak_fma / 1e12:.2f} T FMA/s"
    ctx = capi.Context(0)
    ctx.set_math(False)
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "tiny.bin")
        synth.write_model(path, synth.make_params(synth.TINY, seed=1234))
        model = capi.Model(ctx, open(path, "rb").read())
    model.set_max_length(1024)
    dh = model.E // HEADS
    results = []

    for B, T in SHAPES:
        assert B * T == TOKENS
        batch = Batch(ctx, B, T, seed=T)
        batch.run(model)  # warm-up
        times, tgt = [], 0
        for _ in range(args.reps):
            ctx.flush_l2()
            ctx.timer_start()
            _, t = batch.run(model)
            times.append(ctx.timer_stop())
            tgt += t
        kernels = profiled(ctx, model, batch)
        attn = kernels.get("enc_self_attention", {"ms": float("nan")})
        fmas = 2.0 * B * HEADS * T * T * dh * ENC_LAYERS  # scores + P V over full-length sentences, every encoder layer
        rate = fmas / (attn["ms"] * 1e-3)
        rec = {"shape": f"{B}x{T}", "B": B, "T": T, "math": "exact", "limit_factor": LIMIT, "reps": args.reps,
               "pass_ms": [round(x, 3) for x in times], "target_tok_s": tgt / (sum(times) * 1e-3),
               "self_attention_kernel": "long" if 256 < T <= 384 or T > 556 else "tiled",  # engine.cu's rule
               "self_attention_fma": fmas, "self_attention_ms": attn["ms"], "self_attention_fma_per_s": rate,
               "self_attention_share_of_fp32_fma_peak": rate / peak_fma, "fp32_fma_peak": peak_name,
               "kernels": kernels, **hw}
        print(json.dumps(rec), flush=True)
        results.append(rec)
        batch.free(ctx)

    # tiled vs long self-attention where both fit: event times of the kernel over profiled passes, alternated
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "base.bin")
        synth.write_model(path, synth.make_params(synth.ModelDims(emb=512, ffn=2048, vocab=8000), seed=5))
        base = capi.Model(ctx, open(path, "rb").read())
    base.set_max_length(1024)
    for m, T in [(model, T) for T in AB_T] + [(base, T) for T in AB_T_BASE]:
        dh = m.E // HEADS
        B = TOKENS // T
        batch = Batch(ctx, B, T, seed=T + 1, limit=0.01, vocab=m.V)  # the encoder is what differs; decode one or two steps
        ms = {"tiled": [], "long": []}
        toks = {}
        for kern in ms:
            os.environ["SLIMT_B200_SELFATTN"] = kern
            batch.run(m)  # warm-up
            toks[kern] = ctx.from_device(batch.steps, (batch.max_steps, B), np.uint32)
        for _ in range(args.ab_reps):
            for kern in ms:
                os.environ["SLIMT_B200_SELFATTN"] = kern
                ctx.flush_l2()
                ms[kern].append(profiled(ctx, m, batch)["enc_self_attention"]["ms"])
        del os.environ["SLIMT_B200_SELFATTN"]
        rec = {"ab": f"{B}x{T}", "B": B, "T": T, "head_size": dh, "tiled_ms": ms["tiled"], "long_ms": ms["long"],
               "tiled_median_ms": float(np.median(ms["tiled"])), "long_median_ms": float(np.median(ms["long"])),
               "same_step_tokens": bool(np.array_equal(toks["tiled"], toks["long"])), **hw}
        print(json.dumps(rec), flush=True)
        results.append(rec)
        batch.free(ctx)

    model.close()
    base.close()
    ctx.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for r in results:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
