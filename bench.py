#!/usr/bin/env python
"""bench.py -- headline benchmark of the hot path (BASELINE.json: target tokens/sec, greedy, tiny11 int8).

    python bench.py --gpus N --steps K --warmup W            # our arm (one process per GPU under torchrun for N>1)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's own CPU path (oracle/_ref) on host cores

A "step" is one pass of Model::forward over one batch stream of synthetic input: configs[1] of
BASELINE.json -- tiny11-shaped int8 random-init model with a lexical shortlist, 4096 sentences of 32 tokens
per GPU (weak scaling: every rank owns its own 4096 sentences; sentences are independent, no collective).

Printed JSON (rank 0): `value` = whole-job target tokens/s with the batch resident in HBM (device-timed,
max over ranks); `e2e` = the same metric through the C-ABI call a user makes (slimt_b200_translate: host
buffers, Batcher + shortlist generation on the host, H2D/D2H inside the timed region); `roofline` for the
dominant kernel from per-kernel CUDA-event timings of one extra (untimed) profiled pass; `cpu_baseline`
= the reference compiled in place (oracle/_ref) timed on this box's host cores on a bounded sample.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from slimt_b200 import synth  # noqa: E402

SENTENCES_PER_GPU = 4096
SRC_LEN = 32
LIMIT = 1.5
MODEL_SEED = 1234

# --workload: the headline (default) is BASELINE.json configs[1]; the others are the remaining GPU configs of
# BASELINE.json, benchmarked with the same harness (they are parity-test cases first: tests/test_gpu_model.py).
WORKLOADS = {
    "tiny_shortlist": dict(dims="TINY", shortlist=True, sentences=4096, length=32, max_words=4096 * 32,
                           desc="tiny11 int8 (emb 256, ffn 1536, 6 enc / 2 SSRU dec, vocab 32000, random-init seed 1234) "
                                "with lexical shortlist, greedy decode of 4096 synthetic sentences x 32 tokens per GPU "
                                "(BASELINE.json configs[1])"),
    "tiny_full": dict(dims="TINY", shortlist=False, sentences=4096, length=32, max_words=4096 * 32,
                      desc="tiny11 int8 without shortlist (full 32000-column output GEMM + fused argmax), 4096 synthetic "
                           "sentences x 32 tokens per GPU (BASELINE.json configs[3])"),
    "base_shortlist": dict(dims="BASE", shortlist=True, sentences=4096, length=32, max_words=4096 * 32,
                           desc="base int8 (emb 512, ffn 2048, 6 enc / 2 SSRU dec, vocab 32000, random-init) with lexical "
                                "shortlist, 4096 synthetic sentences x 32 tokens per GPU (BASELINE.json configs[2])"),
    "tiny_b64": dict(dims="TINY", shortlist=True, sentences=64, length=32, max_words=64 * 32,
                     desc="tiny11 int8 with lexical shortlist, ONE batch of 64 synthetic sentences x 32 tokens (BASELINE.json "
                          "configs[0], the reference's CPU-runnable case: the latency regime, two decoder tiles)"),
    "tiny_len64": dict(dims="TINY", shortlist=True, sentences=2048, length=64, max_words=2048 * 64,
                       desc="tiny11 int8 with lexical shortlist, 2048 synthetic sentences x 64 tokens per GPU (the same 131072 "
                            "source tokens as the headline at twice the sentence length: the two-key-block recompute "
                            "cross-attention and the T = 64 fused encoder attention)"),
    "mixed": dict(dims="TINY", shortlist=True, sentences=16384, length=(8, 256), max_words=1 << 20,
                  desc="tiny11 int8 with lexical shortlist, mixed-length sweep: 16384 synthetic sentences per GPU per step, "
                       "lengths U{8..256}, length-bucketed by the Batcher into batches of <= 1048576 padded words "
                       "(BASELINE.json configs[4], per-step slice of the 1M-sentence sweep)"),
}
WL = WORKLOADS["tiny_shortlist"]
# exploration only: SLIMT_B200_BENCH_MAX_WORDS overrides the workload's Batcher limit (the chosen values stay in the table)
_MW = os.environ.get("SLIMT_B200_BENCH_MAX_WORDS")


def wl_dims():
    return getattr(synth, WL["dims"])
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "slimt_ref")


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"], "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe).  nvidia-smi needs a
    moment to start, so the sampler is started before the warm-up; mark() brackets the timed region and only samples
    read inside it count (if the region is too short to contain one, the samples nearest to it -- all taken under the
    same load, warm-up or end-to-end passes -- are used and that is said in `window`)."""

    def __init__(self, index: int):
        self.rows = []  # (host time when read, fields)
        self.proc = None
        self.index = index
        self.t0 = self.t1 = None

    def start(self):
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "10",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.1)
        self.proc.terminate()
        inside = [r for t, r in self.rows if self.t0 is not None and self.t0 <= t <= self.t1 + 0.03]
        window = "timed region"
        if not inside:
            inside = [r for _, r in self.rows]
            window = "warm-up + timed region + end-to-end passes (timed region shorter than one sample)"
        sm, mx, reasons = [], [], set()
        for r in inside:
            try:
                sm.append(float(r[1])), mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": window}


def build_assets(tmp: str, rank: int):
    dims = wl_dims()
    model_path = os.path.join(tmp, "model.bin")
    synth.write_model(model_path, synth.make_params(dims, seed=MODEL_SEED))
    fr, offs, lists = synth.make_shortlist(vocab=dims.vocab, frequent=100, best=100, seed=7)
    sl_path = os.path.join(tmp, "lex.s2t.bin")
    synth.write_shortlist(sl_path, fr, offs, lists, best=100)
    sentences = synth.make_sentences(WL["sentences"], WL["length"], vocab=dims.vocab, seed=1000 + rank)
    return model_path, sl_path, (fr, offs, lists), sentences


def host_isa():
    """What intgemm's RealCPUID (intgemm.cc:40-86) will find on this host: INTGEMM_CPUID requests are capped to it."""
    try:
        flags = next(l for l in open("/proc/cpuinfo") if l.startswith("flags")).split()
    except (OSError, StopIteration):
        return "unknown"
    for name, flag in (("AVX512VNNI", "avx512_vnni"), ("AVX512BW", "avx512bw"), ("AVX2", "avx2"), ("SSSE3", "ssse3")):
        if flag in flags:
            return name
    return "SSE2"


def cpu_sample(sentences, cores):
    """A bounded sample of the workload for the CPU arm: one batch per host thread, sized so a pass takes seconds.
    Returns (sentences, sentences per batch)."""
    long_ones = not isinstance(WL["length"], int) or WL["length"] > 64
    per_batch = 8 if long_ones else 64
    n = min(len(sentences), per_batch * cores)
    return sentences[:n], per_batch


def cpu_reference_run(model_path, shortlist, sentences, workers, batch_sentences=64, repeats=1, isa=None, want_tokens=False):
    """Times oracle/_ref/slimt_ref (the unmodified reference, intgemm provider) on `workers` host threads.  `isa`
    sets INTGEMM_CPUID (intgemm.cc:90-108): AVX512VNNI = exact int32 accumulation, AVX512BW = the maddubs path with
    int16 pair saturation, the arithmetic of slimt's default gemmology provider."""
    from oracle import slimt_oracle as so
    fr, offs, lists = shortlist
    nb = max(1, (len(sentences) + batch_sentences - 1) // batch_sentences)
    recs = []
    for b in range(nb):
        chunk = sentences[b * batch_sentences:(b + 1) * batch_sentences]
        words = np.concatenate(chunk)
        sl = so.shortlist_generate(words, fr, offs, lists, wl_dims().vocab) if WL["shortlist"] else None
        recs.append(synth.pack_batch(chunk, LIMIT, sl))
    with tempfile.NamedTemporaryFile(suffix=".batches", delete=False) as f:
        f.write(np.uint32(len(recs)).tobytes() + b"".join(recs))
        path = f.name
    tok_path = path + ".tokens"
    env = dict(os.environ)
    if isa:
        env["INTGEMM_CPUID"] = isa
    try:
        cmd = [REF_BIN, "bench", "--model", model_path, "--batches", path, "--workers", str(workers), "--repeat", str(repeats)]
        if want_tokens:
            cmd += ["--tokens-out", tok_path]
        out = subprocess.run(cmd, capture_output=True, text=True, check=True, env=env).stdout
        tokens = None
        if want_tokens:
            flat = np.fromfile(tok_path, dtype=np.uint32)
            tokens, p = [], 1
            for _ in range(int(flat[0])):
                nbs = int(flat[p])
                p += 1
                for _ in range(nbs):
                    n = int(flat[p])
                    tokens.append(flat[p + 1:p + 1 + n])
                    p += 1 + n
    finally:
        os.unlink(path)
        if os.path.exists(tok_path):
            os.unlink(tok_path)
    lines = [json.loads(l) for l in out.strip().splitlines()]
    return (lines, tokens) if want_tokens else lines


def cpu_baseline_block(model_path, shortlist, sentences, repeats=2):
    """cpu_baseline of the bench line: the reference on all host threads, on a bounded sample, for both intgemm code
    paths BASELINE.md section 4.4 asks for.  The headline row is the exact one (VNNI when the host has it)."""
    cores = os.cpu_count() or 1
    sample, per_batch = cpu_sample(sentences, cores)
    rows, toks = [], {}
    for isa in ("AVX512VNNI", "AVX512BW"):
        lines, tokens = cpu_reference_run(model_path, shortlist, sample, cores, per_batch, repeats, isa=isa, want_tokens=True)
        best = max(lines, key=lambda l: l["target_tokens_per_s"])
        rows.append({"isa_requested": isa, "value": best["target_tokens_per_s"], "unit": "tokens/s",
                     "seconds": best["seconds"], "target_tokens": best["target_tokens"]})
        toks[isa] = tokens
    a, b = toks["AVX512VNNI"], toks["AVX512BW"]
    same_sent = sum(1 for x, y in zip(a, b) if len(x) == len(y) and np.array_equal(x, y))
    same_tok = sum(int((x[:min(len(x), len(y))] == y[:min(len(x), len(y))]).sum()) for x, y in zip(a, b))
    all_tok = sum(max(len(x), len(y)) for x, y in zip(a, b))
    lens = WL["length"] if isinstance(WL["length"], int) else f"{WL['length'][0]}-{WL['length'][1]}"
    return {
        "value": rows[0]["value"], "unit": "tokens/s", "cores": cores, "kind": "reference",
        "sample": f"{len(sample)} of {WL['sentences']} sentences (lengths {lens}) in {per_batch}-sentence batches"
                  f"{' each with its own shortlist union' if WL['shortlist'] else ''}, one batch per host thread, best of "
                  f"{repeats}; oracle/_ref = the unmodified reference compiled in place, intgemm provider + ruy sgemm "
                  f"(gemmology needs xsimd: unbuildable offline)",
        "host_isa": host_isa(),
        "rows": rows,
        "saturation": {"note": "AVX512BW = maddubs with int16 pair saturation (gemmology-equivalent arithmetic) against "
                               "AVX512VNNI = exact int32 accumulation (what the GPU computes); requests above host_isa are capped",
                       "sentences_identical": same_sent, "sentences": len(a),
                       "token_agreement": round(same_tok / max(1, all_tok), 6)},
    }


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    tmp = tempfile.mkdtemp(prefix="slimt_b200_ref_")
    model_path, _, shortlist, sentences = build_assets(tmp, 0)
    if not os.path.exists(REF_BIN):
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/slimt_ref not built (needs /root/reference)"}))
        return 0
    # Each step is a bounded sample of the workload: one batch per host thread (the reference's Async model,
    # Frontend.cc:207-227: `workers` threads, each running Model::forward on its own batch).
    sample, per_batch = cpu_sample(sentences, cores)
    lines = cpu_reference_run(model_path, shortlist, sample, cores, per_batch, repeats=args.warmup + args.steps)
    timed = lines[args.warmup:]
    secs = sum(l["seconds"] for l in timed)
    toks = sum(l["target_tokens"] for l in timed)
    value = toks / secs
    lens = WL["length"] if isinstance(WL["length"], int) else f"{WL['length'][0]}-{WL['length'][1]}"
    sample_desc = (f"{len(sample)} of {WL['sentences']} sentences (lengths {lens}) per step in {per_batch}-sentence batches"
                   f"{', each with its own shortlist union (smaller than the GPU arm\'s whole-batch union)' if WL['shortlist'] else ''}"
                   f", one batch per host thread; intgemm provider (host ISA {host_isa()}), ruy sgemm")
    cfg = workload_config()
    cfg["reference_batching"] = {"sentences_per_batch": per_batch, "batches_per_step": (len(sample) + per_batch - 1) // per_batch,
                                 "threads": cores}
    print(json.dumps({
        "impl": "reference", "metric": "target_tokens_per_sec", "value": value, "unit": "tokens/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / max(1, len(timed)),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int8", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": value, "unit": "tokens/s", "cores": cores, "kind": "reference", "sample": sample_desc},
        "e2e": {"value": value, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))
    return 0


def run_single_process(args):
    """One process, one Batcher, N GPUs: slimt_b200_translate_multi deals the request's batches to one model replica
    per GPU (two lanes each).  This is the service shape of the reference's Async (Frontend.cc:207-227) and the
    measurement of SURVEY.md section 8(e)'s scaling risk: ONE host feeding N GPUs.  `value` is end to end by
    construction (host buffers in and out); strong scaling: the request is the same for every N."""
    import ctypes
    from slimt_b200 import capi
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    n_sent = args.sentences or WL["sentences"]
    dims = wl_dims()
    tmp = tempfile.mkdtemp(prefix="slimt_b200_sp_")
    model_path = os.path.join(tmp, "model.bin")
    synth.write_model(model_path, synth.make_params(dims, seed=MODEL_SEED))
    fr, offs, lists = synth.make_shortlist(vocab=dims.vocab, frequent=100, best=100, seed=7)
    sl_path = os.path.join(tmp, "lex.s2t.bin")
    synth.write_shortlist(sl_path, fr, offs, lists, best=100)
    t0 = time.perf_counter()
    rng = np.random.RandomState(1000)
    if isinstance(WL["length"], int):
        lens = np.full(n_sent, WL["length"], dtype=np.int64)
    else:
        lens = rng.randint(WL["length"][0], WL["length"][1] + 1, size=n_sent).astype(np.int64)
    h_offsets = np.zeros(n_sent + 1, dtype=np.uint64)
    h_offsets[1:] = np.cumsum(lens)
    h_tokens = rng.randint(1, dims.vocab, size=int(h_offsets[-1])).astype(np.uint32)
    h_tokens[(h_offsets[1:] - 1).astype(np.int64)] = synth.EOS_ID  # every sentence ends in EOS
    gen_s = time.perf_counter() - t0
    blob = open(model_path, "rb").read()
    ctxs = [capi.Context(i) for i in range(args.gpus)]
    for c in ctxs:
        c.set_math(args.math == "fast")
    models = [capi.Model(c, blob) for c in ctxs]
    sl_bin = open(sl_path, "rb").read() if WL["shortlist"] else None
    sl_buf = (ctypes.c_char * len(sl_bin)).from_buffer_copy(sl_bin) if sl_bin is not None else None
    max_steps = max(1, int(np.float32(LIMIT) * np.float32(lens.max())))
    out_tokens = np.zeros(int(n_sent) * max_steps, dtype=np.uint32)
    out_offsets = np.zeros(n_sent + 1, dtype=np.uint64)
    sampler = ClockSampler(0)
    sampler.start()
    # warm-up: a slice of the request, enough to build every lane's workspace and touch every kernel variant
    warm = min(n_sent, 4096 * args.gpus)
    for _ in range(max(1, args.warmup - 2)):
        models[0].translate_flat(h_tokens[:int(h_offsets[warm])], h_offsets[:warm + 1], WL["max_words"], LIMIT, sl_buf,
                                 out_tokens, out_offsets[:warm + 1], replicas=models)
    sampler.mark_begin()
    secs, toks, st = 0.0, 0, None
    steps = max(1, args.steps)
    for _ in range(steps):
        t0 = time.perf_counter()
        _, _, st = models[0].translate_flat(h_tokens, h_offsets, WL["max_words"], LIMIT, sl_buf, out_tokens, out_offsets,
                                            replicas=models)
        secs += time.perf_counter() - t0
        toks += st["target_tokens"]
    sampler.mark_end()
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {f"{args.math}_tokens": out_tokens[:int(out_offsets[-1])].astype(np.float32),
                                         f"{args.math}_offsets": out_offsets.astype(np.float64)})
    cfg = workload_config()
    cfg["sentences_per_gpu"] = None
    cfg["sentences"] = int(n_sent)
    cfg["sharding"] = ("one process: one Batcher, batches dealt to one replica per GPU (slimt_b200_translate_multi), two lanes per "
                       "replica; no collective")
    cfg["l2"] = "inputs larger than L2 (a fresh batch every forward pass)"
    value = toks / secs
    out = {"metric": "target_tokens_per_sec", "value": value, "unit": "tokens/s", "n_gpus": args.gpus, "steps": steps,
           "warmup": args.warmup, "ms_per_step": 1e3 * secs / steps, "higher_is_better": True, "scaling": "strong",
           "vs_baseline": None, "dtype": "int8", "data": "synthetic", "config": cfg, "clocks": clocks, "math": args.math,
           "mode": "single-process", "e2e": {"value": value, "unit": "tokens/s", "h2d_bytes_per_step": st["h2d_bytes"],
                                             "d2h_bytes_per_step": st["d2h_bytes"],
                                             "api": "slimt_b200_translate_multi (host buffers, one call per step)"},
           "gpu_launches": st["kernel_launches"] * steps, "batches_per_step": st["batches"],
           "device_ms_longest_replica": st["device_ms"], "host_cores": os.cpu_count(),
           "input_generation_s": round(gen_s, 2)}
    os.write(json_fd, (json.dumps(out) + "\n").encode())
    return 0


DUMP_CAP_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Writes each array as out_dir/<name>.npy.  Beyond DUMP_CAP_BYTES in all, every array is replaced by a fixed, seeded
    sample of its elements (in order), so two builds run with the same arguments still compare element for element."""
    os.makedirs(out_dir, exist_ok=True)
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        if total > DUMP_CAP_BYTES:
            a = a.ravel()[np.sort(np.random.RandomState(0).choice(a.size, a.size * DUMP_CAP_BYTES // total, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)
    print(f"bench: wrote {len(arrays)} arrays to {out_dir}" + (" (sampled)" if total > DUMP_CAP_BYTES else ""), file=sys.stderr)


def workload_config():
    return {"workload": WL["desc"], "sentences_per_gpu": WL["sentences"], "src_len": WL["length"], "limit_factor": LIMIT,
            "max_words": WL["max_words"], "l2": "flushed between timed steps (256 MiB memset)",
            "sharding": "independent sentences per rank, no collective"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200,
                    help="timed passes; the default keeps the timed region above 2 s at the headline size")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="tiny_shortlist", choices=sorted(WORKLOADS),
                    help="tiny_shortlist = the headline (BASELINE.json configs[1]); the others are its remaining GPU configs")
    ap.add_argument("--math", default="both", choices=["both", "fast", "exact"],
                    help="arithmetic mode(s) to measure; with `both` the top-level keys are the bit-exact mode's and the "
                         "tolerance mode's numbers are reported beside them under `fast`")
    ap.add_argument("--single-process", action="store_true",
                    help="serve ONE request with --gpus replicas from this process (slimt_b200_translate_multi) instead of "
                         "one process per GPU; strong scaling")
    ap.add_argument("--sentences", type=int, default=0, help="with --single-process: sentences in the request (default: the workload's)")
    ap.add_argument("--profiler-range", action="store_true",
                    help="bracket the timed steps with cudaProfilerStart/Stop (for ncu --profile-from-start off)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned to the caller as DIR/<name>.npy "
                         "(token ids as float32, offsets as float64; rank 0; at most 64 MiB, a seeded sample beyond that)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of this project's GPU path, not of --impl reference")
    global WL
    WL = dict(WORKLOADS[args.workload])
    if _MW:
        WL["max_words"] = int(_MW)
        WL["desc"] += f" [max_words overridden to {_MW}]"
    if args.impl == "reference":
        return run_reference_arm(args)
    if args.single_process:
        if args.math == "both":
            args.math = "exact"
        return run_single_process(args)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    dist = None
    # stdout carries exactly one JSON line: native libraries that write to fd 1 (NCCL's version banner) go to stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl")

    from slimt_b200 import capi
    ctx = capi.Context(local_rank)  # raises without a GPU: no CPU fallback
    tmp = tempfile.mkdtemp(prefix=f"slimt_b200_bench_{rank}_")
    model_path, sl_path, shortlist, sentences = build_assets(tmp, rank)
    model = capi.Model(ctx, open(model_path, "rb").read())
    sl_bin = open(sl_path, "rb").read() if WL["shortlist"] else None
    max_words = WL["max_words"]

    # ---- device-resident arm: the batches a Batcher would form, uploaded once
    plan = capi.batcher_plan([len(s) for s in sentences], max_words)
    resident = []
    for ids, width in plan:
        B = len(ids)
        tok = np.zeros((B, width), dtype=np.uint32)
        lens = np.zeros(B, dtype=np.uint32)
        for r, i in enumerate(ids):
            tok[r, :len(sentences[i])] = sentences[i]
            lens[r] = len(sentences[i])
        max_steps = max(1, int(np.float32(LIMIT) * np.float32(width)))
        entry = {"B": B, "T": width, "tok": ctx.to_device(tok), "lens": ctx.to_device(lens), "sl": None, "nsl": 0,
                 "steps": ctx.dev_alloc(4 * max_steps * B)}
        if sl_bin is not None:
            sl = capi.shortlist_generate(sl_bin, np.concatenate([sentences[i] for i in ids]), model.V)
            entry["sl"], entry["nsl"] = ctx.to_device(sl), len(sl)
        resident.append(entry)

    def resident_pass():
        toks = 0
        for b in resident:
            b["decode_steps"], t = model.forward_resident(b["tok"], b["lens"], b["B"], b["T"], b["steps"], LIMIT, b["sl"], b["nsl"])
            toks += t
        return toks

    def barrier():
        ctx.synchronize()
        if dist is not None:
            dist.barrier()

    def step_tokens_of(entry):
        steps = max(1, int(np.float32(LIMIT) * np.float32(entry["T"])))
        return ctx.from_device(entry["steps"], (steps, entry["B"]), np.uint32)

    import ctypes
    h_offsets = np.zeros(len(sentences) + 1, dtype=np.uint64)
    h_offsets[1:] = np.cumsum([len(s) for s in sentences])
    h_tokens = np.concatenate([np.asarray(s, dtype=np.uint32) for s in sentences])
    h_out_tokens = np.zeros(len(sentences) * (int(LIMIT * max(len(s) for s in sentences)) + 1), dtype=np.uint32)
    h_out_offsets = np.zeros(len(sentences) + 1, dtype=np.uint64)
    sl_buf = (ctypes.c_char * len(sl_bin)).from_buffer_copy(sl_bin) if sl_bin is not None else None

    peaks = measured_peaks()
    # int8 dense denominator: SURVEY.md section 6 asks for max(measured int8, 2 x measured bf16).  The int8 figure is
    # our own tcgen05 kind::i8 issue-rate measurement on this pool's B200 (tools/mma_peak.cu -> profiles/).
    int8_peak_tops, int8_src = 2.0 * peaks["bf16_tflops"], f"2 x {peaks['source']} bf16 burst ({peaks['bf16_tflops']} TF/s)"
    mma_path = os.path.join(ROOT, "profiles", "r1_mma_i8_peak.jsonl")
    if os.path.exists(mma_path):
        rows = [json.loads(l) for l in open(mma_path) if l.strip()]
        best = max((r.get("tops_all_sms", 0.0) for r in rows), default=0.0)
        if best > int8_peak_tops:
            int8_peak_tops, int8_src = best, "measured tcgen05 kind::i8 128x256x32 issue rate, 148 SMs (profiles/r1_mma_i8_peak.jsonl)"
    traffic = {}
    tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tpath):
        traffic = json.load(open(tpath))  # kernel tag -> dram bytes (read + write) per launch, from ncu --set full

    def measure(mode, sampler=None):
        """One full measurement (device-resident arm, end-to-end arm, per-kernel pass) in one arithmetic mode."""
        ctx.set_math(mode == "fast")
        for _ in range(args.warmup):
            resident_pass()
        barrier()
        if sampler:
            sampler.mark_begin()
        launches0 = ctx.launches()
        step_ms, tokens_per_step = [], 0
        if args.profiler_range:
            import torch
            torch.cuda.cudart().cudaProfilerStart()
        for _ in range(args.steps):
            ctx.flush_l2()
            ctx.timer_start()
            tokens_per_step = resident_pass()
            step_ms.append(ctx.timer_stop())
        launches = ctx.launches() - launches0
        if args.profiler_range:
            ctx.synchronize()
            torch.cuda.cudart().cudaProfilerStop()
        barrier()
        if sampler:
            sampler.mark_end()
        total_ms = sum(step_ms)
        tokens = [step_tokens_of(e) for e in resident]
        outputs = {}
        if args.dump_outputs:  # per batch of the plan: step tokens [decode steps, sentences of the batch]
            outputs = {f"{mode}_step_tokens_{i:03d}": t[:e["decode_steps"]].astype(np.float32)
                       for i, (e, t) in enumerate(zip(resident, tokens))}

        # ---- end-to-end arm through the public C-ABI call with host buffers (ragged tokens/offsets in, ragged targets
        # out; Batcher, shortlist generation, H2D and D2H all inside the timed call)
        for _ in range(max(1, args.warmup - 1)):
            model.translate_flat(h_tokens, h_offsets, max_words, LIMIT, sl_buf, h_out_tokens, h_out_offsets)
        barrier()
        e2e_s, e2e_tokens, e2e_stats = 0.0, 0, None
        for _ in range(args.steps):
            t0 = time.perf_counter()
            _, _, st = model.translate_flat(h_tokens, h_offsets, max_words, LIMIT, sl_buf, h_out_tokens, h_out_offsets)
            e2e_s += time.perf_counter() - t0
            e2e_tokens += st["target_tokens"]
            e2e_stats = st
        barrier()
        if args.dump_outputs:
            outputs[f"{mode}_e2e_tokens"] = h_out_tokens[:int(h_out_offsets[-1])].astype(np.float32)
            outputs[f"{mode}_e2e_offsets"] = h_out_offsets.astype(np.float64)

        # ---- per-kernel event timing: one extra profiled pass (not part of the timed region)
        ctx.profile(True)
        resident_pass()
        stats = ctx.profile_read()
        ctx.profile(False)

        if dist is not None:
            import torch
            t = torch.tensor([total_ms, e2e_s], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            total_ms, e2e_s = float(t[0]), float(t[1])
            n = torch.tensor([float(tokens_per_step * args.steps), float(e2e_tokens), float(launches)], dtype=torch.float64, device="cuda")
            dist.all_reduce(n, op=dist.ReduceOp.SUM)
            all_tokens, all_e2e_tokens, all_launches = float(n[0]), float(n[1]), int(n[2])
        else:
            all_tokens, all_e2e_tokens, all_launches = float(tokens_per_step * args.steps), float(e2e_tokens), launches

        kern = []
        tot_prof_ms = sum(s["ms"] for s in stats) or 1.0
        for s in sorted(stats, key=lambda s: -s["ms"]):
            sec = s["ms"] * 1e-3
            entry = {"name": s["name"], "launches": s["launches"], "ms": round(s["ms"], 4), "share": round(s["ms"] / tot_prof_ms, 4),
                     "avg_us": round(1e3 * s["ms"] / max(1, s["launches"]), 2)}
            if s["ops"] > 0:
                entry["tops"] = round(s["ops"] / sec / 1e12, 2)
                entry["tensor_frac"] = round(s["ops"] / sec / 1e12 / int8_peak_tops, 4)
            entry["gbs"] = round(s["bytes"] / sec / 1e9, 1)
            entry["hbm_frac"] = round(s["bytes"] / sec / 1e9 / peaks["hbm_gbs"], 4)
            kern.append(entry)
        top = kern[0]
        top_raw = next(s for s in stats if s["name"] == top["name"])
        tensor_bound = top.get("tensor_frac", 0) > top["hbm_frac"]
        if tensor_bound:
            roof = {"kernel": top["name"], "bound": "tensor", "achieved": top["tops"], "peak": int8_peak_tops, "unit": "TOP/s",
                    "frac": top["tensor_frac"], "traffic": traffic.get(top["name"]), "peak_source": int8_src}
        else:
            roof = {"kernel": top["name"], "bound": "hbm", "achieved": top["gbs"], "peak": peaks["hbm_gbs"], "unit": "GB/s",
                    "frac": top["hbm_frac"], "traffic": traffic.get(top["name"]), "peak_source": f"{peaks['source']} copy bandwidth"}
        roof["algorithmic_per_launch"] = (top_raw["ops"] if tensor_bound else top_raw["bytes"]) / max(1, top_raw["launches"])
        roof["avg_launch_us"] = top["avg_us"]
        roof["share_of_step"] = top["share"]
        gemm_ops = sum(s["ops"] for s in stats)
        gemm_ms = sum(s["ms"] for s in stats if s["ops"] > 0)
        return {
            "math": mode, "value": all_tokens / (total_ms * 1e-3), "ms_per_step": total_ms / args.steps,
            "e2e": {"value": all_e2e_tokens / e2e_s, "unit": "tokens/s", "h2d_bytes_per_step": e2e_stats["h2d_bytes"],
                    "d2h_bytes_per_step": e2e_stats["d2h_bytes"], "api": "slimt_b200_translate (host buffers)"},
            "gpu_launches": all_launches, "roofline": roof, "kernels": kern,
            "int8_gemm_summary": {"algorithmic_tops": round(gemm_ops / 1e12, 3), "ms_in_gemm_kernels": round(gemm_ms, 3),
                                  "achieved_tops": round(gemm_ops / max(gemm_ms, 1e-9) / 1e9, 1), "peak_tops": int8_peak_tops,
                                  "frac": round(gemm_ops / max(gemm_ms, 1e-9) / 1e9 / int8_peak_tops, 4),
                                  "note": "all kernels that issue tcgen05 MMAs, fused epilogues included in their time"},
            "target_tokens_per_step_per_gpu": tokens_per_step, "_tokens": tokens, "_outputs": outputs,
        }

    sampler = ClockSampler(local_rank)
    sampler.start()
    modes = ["exact", "fast"] if args.math == "both" else [args.math]
    res = {}
    for i, mode in enumerate(modes):
        res[mode] = measure(mode, sampler if i == 0 else None)
    clocks = sampler.stop()
    ctx.set_math(False)

    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return 0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {k: v for m in modes for k, v in res[m]["_outputs"].items()})

    head = res[modes[0]]
    out = {
        "metric": "target_tokens_per_sec", "value": head["value"], "unit": "tokens/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "int8", "data": "synthetic", "config": workload_config(),
        "clocks": clocks, "math": head["math"],
        "e2e": head["e2e"], "gpu_launches": head["gpu_launches"], "roofline": head["roofline"], "kernels": head["kernels"],
        "int8_gemm_summary": head["int8_gemm_summary"],
        "target_tokens_per_step_per_gpu": head["target_tokens_per_step_per_gpu"],
        "batches_per_step": len(resident),
    }
    out["config"]["math"] = (
        "exact = every float bit-identical to the reference CPU path (intgemm, exact int32 accumulation); the default and the "
        "mode all top-level numbers are measured in" if head["math"] == "exact" else
        "fast = tolerance mode: f32/int32 arithmetic throughout, FMA-contracted dequantisation, tree-reduced LayerNorm sums, "
        "ex2/rcp softmax and sigmoid, integer argmax proxy (tests/test_gpu_fast_mode.py says what that costs in agreement)")
    if len(modes) == 2:
        other = res[modes[1]]
        out[other["math"]] = {k: other[k] for k in ("value", "ms_per_step", "e2e", "gpu_launches", "roofline", "int8_gemm_summary", "kernels")}
        same = sum(int((x == y).sum()) for x, y in zip(head["_tokens"], other["_tokens"]))
        total = sum(x.size for x in head["_tokens"])
        # a sentence counts as identical when every step token agrees (one early difference changes all later inputs)
        sent_same = sum(int((x == y).all(axis=0).sum()) for x, y in zip(head["_tokens"], other["_tokens"]))
        sent_total = sum(x.shape[1] for x in head["_tokens"])
        out["fast_vs_exact"] = {"step_tokens_equal": round(same / max(1, total), 6), "sentences_identical": round(sent_same / max(1, sent_total), 6),
                                "note": "greedy free-running decode of this run's own batch in both modes (rank 0); exact mode equals the "
                                        "reference token for token (tests/test_gpu_large_golden.py); in tolerance mode a few-ulp "
                                        "difference occasionally moves one int8 operand by one step, which this random-init model "
                                        "amplifies, and a sentence that differs once differs in all later tokens"}

    if not args.no_cpu_baseline:
        if os.path.exists(REF_BIN):
            out["cpu_baseline"] = cpu_baseline_block(model_path, shortlist, sentences)
        else:
            from oracle import slimt_oracle as so
            fr, offs, lists = shortlist
            chunk = sentences[:16]
            tok = np.zeros((16, max(len(s) for s in chunk)), dtype=np.uint32)
            for i, s in enumerate(chunk):
                tok[i, :len(s)] = s
            sl = so.shortlist_generate(np.concatenate(chunk), fr, offs, lists, wl_dims().vocab) if WL["shortlist"] else None
            orc = so.Oracle(synth.read_model(model_path))
            t0 = time.perf_counter()
            res = orc.forward(tok, np.array([len(s) for s in chunk]), LIMIT, shortlist=sl)
            dt = time.perf_counter() - t0
            out["cpu_baseline"] = {"value": sum(len(s) for s in res["sentences"]) / dt, "unit": "tokens/s", "cores": 1,
                                   "kind": "port", "sample": "16 sentences through oracle/slimt_oracle.py (oracle/_ref not built)"}
    os.write(json_fd, (json.dumps(out) + "\n").encode())
    return 0


if __name__ == "__main__":
    sys.exit(main())
