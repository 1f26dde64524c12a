"""ctypes view of the C ABI in include/slimt_b200.h, used by tests/ and bench.py.

This is harness code: the product is the shared library (CUDA kernels + host
C++).  Loading fails loudly when the library is missing; creating a context
fails loudly without a CUDA device -- there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# SLIMT_B200_LIB selects another build of the same library (A/B measurements of kernel variants)
LIB_PATH = os.environ.get("SLIMT_B200_LIB") or os.path.join(_HERE, "libslimt_b200.so")
_lib = None

EXPORTS = [
    "slimt_b200_last_error", "slimt_b200_version", "slimt_b200_ctx_create", "slimt_b200_ctx_destroy",
    "slimt_b200_ctx_synchronize", "slimt_b200_dev_alloc", "slimt_b200_dev_free", "slimt_b200_memcpy_h2d",
    "slimt_b200_memcpy_d2h", "slimt_b200_timer_start", "slimt_b200_timer_stop", "slimt_b200_flush_l2",
    "slimt_b200_qmm_prepare_weight_quantized_transposed", "slimt_b200_qmm_prepare_weight_transposed",
    "slimt_b200_qmm_affine", "slimt_b200_qmm_affine_debug", "slimt_b200_model_create", "slimt_b200_model_destroy",
    "slimt_b200_model_dims", "slimt_b200_model_forward", "slimt_b200_translate", "slimt_b200_kernel_launches",
    "slimt_b200_shortlist_generate", "slimt_b200_batcher_plan", "slimt_b200_profile_enable", "slimt_b200_profile_read",
    "slimt_b200_translate_multi", "slimt_b200_shortlist_check", "slimt_b200_ctx_set_math", "slimt_b200_ctx_get_math",
    "slimt_b200_model_set_max_length", "slimt_b200_model_max_length",
]


class ModelConfig(C.Structure):
    _fields_ = [("encoder_layers", C.c_int32), ("decoder_layers", C.c_int32), ("feed_forward_depth", C.c_int32),
                ("num_heads", C.c_int32), ("eos_id", C.c_uint32), ("pad_id", C.c_uint32)]


class ForwardIO(C.Structure):
    _fields_ = [("tokens", C.c_void_p), ("lengths", C.c_void_p), ("batch", C.c_size_t), ("seq", C.c_size_t),
                ("limit_factor", C.c_float), ("shortlist", C.c_void_p), ("n_shortlist", C.c_size_t),
                ("forced", C.c_void_p), ("device_io", C.c_int32), ("step_tokens", C.c_void_p), ("steps", C.c_size_t),
                ("target_tokens", C.c_uint64), ("encoder_out", C.c_void_p), ("logits", C.c_void_p),
                ("alignment", C.c_void_p)]


class TranslateIO(C.Structure):
    _fields_ = [("tokens", C.c_void_p), ("offsets", C.c_void_p), ("n_sentences", C.c_size_t),
                ("max_words", C.c_size_t), ("limit_factor", C.c_float), ("shortlist_bin", C.c_void_p),
                ("shortlist_bytes", C.c_size_t), ("shortlist_check", C.c_int32), ("shortlist_shared", C.c_int32),
                ("out_tokens", C.c_void_p), ("out_capacity", C.c_size_t), ("out_offsets", C.c_void_p),
                ("out_alignments", C.c_void_p), ("align_capacity", C.c_size_t), ("out_align_offsets", C.c_void_p),
                ("target_tokens", C.c_uint64), ("batches", C.c_uint64),
                ("device_ms", C.c_double), ("kernel_launches", C.c_uint64), ("h2d_bytes", C.c_uint64),
                ("d2h_bytes", C.c_uint64)]


class KernelStat(C.Structure):
    _fields_ = [("name", C.c_char * 48), ("launches", C.c_uint64), ("ms", C.c_double), ("ops", C.c_double),
                ("bytes", C.c_double)]


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(make -C slimt_b200/csrc); there is no fallback path")
        L = C.CDLL(LIB_PATH)
        L.slimt_b200_last_error.restype = C.c_char_p
        L.slimt_b200_version.restype = C.c_char_p
        L.slimt_b200_dev_alloc.restype = C.c_void_p
        L.slimt_b200_dev_alloc.argtypes = [C.c_void_p, C.c_size_t]
        L.slimt_b200_dev_free.argtypes = [C.c_void_p, C.c_void_p]
        L.slimt_b200_memcpy_h2d.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
        L.slimt_b200_memcpy_d2h.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
        L.slimt_b200_ctx_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        L.slimt_b200_ctx_destroy.argtypes = [C.c_void_p]
        L.slimt_b200_ctx_synchronize.argtypes = [C.c_void_p]
        L.slimt_b200_ctx_set_math.argtypes = [C.c_void_p, C.c_int]
        L.slimt_b200_ctx_get_math.argtypes = [C.c_void_p]
        L.slimt_b200_timer_start.argtypes = [C.c_void_p]
        L.slimt_b200_timer_stop.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
        L.slimt_b200_flush_l2.argtypes = [C.c_void_p, C.c_size_t]
        L.slimt_b200_kernel_launches.argtypes = [C.c_void_p]
        L.slimt_b200_kernel_launches.restype = C.c_uint64
        L.slimt_b200_qmm_affine_debug.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p, C.c_size_t,
                                                  C.c_void_p, C.c_float, C.c_float, C.c_void_p, C.c_size_t, C.c_void_p,
                                                  C.c_void_p, C.c_void_p]
        L.slimt_b200_qmm_affine.argtypes = L.slimt_b200_qmm_affine_debug.argtypes[:12]
        L.slimt_b200_qmm_prepare_weight_quantized_transposed.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t]
        L.slimt_b200_qmm_prepare_weight_transposed.argtypes = [C.c_void_p, C.c_void_p, C.c_float, C.c_size_t, C.c_size_t]
        L.slimt_b200_model_create.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(ModelConfig),
                                              C.POINTER(C.c_void_p)]
        L.slimt_b200_model_destroy.argtypes = [C.c_void_p]
        L.slimt_b200_model_dims.argtypes = [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
        L.slimt_b200_model_set_max_length.argtypes = [C.c_void_p, C.c_int32]
        L.slimt_b200_model_max_length.argtypes = [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
        L.slimt_b200_model_forward.argtypes = [C.c_void_p, C.POINTER(ForwardIO)]
        L.slimt_b200_translate.argtypes = [C.c_void_p, C.POINTER(TranslateIO)]
        L.slimt_b200_translate_multi.argtypes = [C.POINTER(C.c_void_p), C.c_size_t, C.POINTER(TranslateIO)]
        L.slimt_b200_shortlist_check.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t]
        L.slimt_b200_shortlist_generate.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p,
                                                    C.c_size_t, C.POINTER(C.c_size_t)]
        L.slimt_b200_batcher_plan.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p,
                                              C.POINTER(C.c_size_t)]
        L.slimt_b200_profile_enable.argtypes = [C.c_void_p, C.c_int]
        L.slimt_b200_profile_read.argtypes = [C.c_void_p, C.POINTER(KernelStat), C.c_size_t, C.POINTER(C.c_size_t)]
        _lib = L
    return _lib


def shortlist_generate(shortlist_bin: bytes, words: np.ndarray, vocab: int) -> np.ndarray:
    """ShortlistGenerator::generate through the C ABI (host only, no GPU needed)."""
    words = np.ascontiguousarray(words, dtype=np.uint32)
    out = np.empty(vocab + 8, dtype=np.uint32)
    n = C.c_size_t()
    buf = (C.c_char * len(shortlist_bin)).from_buffer_copy(shortlist_bin)
    _check(lib().slimt_b200_shortlist_generate(buf, len(shortlist_bin), _ptr(words), len(words), vocab, _ptr(out), len(out),
                                               C.byref(n)), "slimt_b200_shortlist_generate")
    return out[:n.value].copy()


def shortlist_check(shortlist_bin: bytes, vocab: int) -> None:
    """ShortlistGenerator::load with check = true (checksum + content_check); raises on a bad image."""
    buf = (C.c_char * len(shortlist_bin)).from_buffer_copy(shortlist_bin)
    _check(lib().slimt_b200_shortlist_check(buf, len(shortlist_bin), vocab), "slimt_b200_shortlist_check")


def batcher_plan(lengths, max_words: int):
    """Batcher::generate through the C ABI (host only). Returns [(sentence ids, padded width)]."""
    lengths = np.ascontiguousarray(lengths, dtype=np.uint64)
    n = len(lengths)
    ids = np.zeros(max(n, 1), dtype=np.uint64)
    offs = np.zeros(n + 1, dtype=np.uint64)
    widths = np.zeros(max(n, 1), dtype=np.uint64)
    nb = C.c_size_t()
    _check(lib().slimt_b200_batcher_plan(_ptr(lengths), n, max_words, _ptr(ids), _ptr(offs), _ptr(widths), C.byref(nb)),
           "slimt_b200_batcher_plan")
    return [(ids[int(offs[i]):int(offs[i + 1])].astype(np.int64), int(widths[i])) for i in range(nb.value)]


def _err() -> str:
    return lib().slimt_b200_last_error().decode()


def _check(rc: int, what: str) -> None:
    if rc != 0:
        raise RuntimeError(f"{what} failed: {_err()}")


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class Context:
    def __init__(self, device: int = 0):
        self.h = C.c_void_p()
        _check(lib().slimt_b200_ctx_create(device, C.byref(self.h)), "slimt_b200_ctx_create")

    def close(self):
        if self.h:
            lib().slimt_b200_ctx_destroy(self.h)
            self.h = C.c_void_p()

    def synchronize(self):
        _check(lib().slimt_b200_ctx_synchronize(self.h), "synchronize")

    def set_math(self, fast: bool):
        """False: bit-exact mode (default).  True: tolerance mode (logits rtol 1e-3, >= 99 % tokens)."""
        _check(lib().slimt_b200_ctx_set_math(self.h, int(fast)), "set_math")

    def math(self) -> str:
        return "fast" if lib().slimt_b200_ctx_get_math(self.h) else "exact"

    def launches(self) -> int:
        return int(lib().slimt_b200_kernel_launches(self.h))

    def timer_start(self):
        _check(lib().slimt_b200_timer_start(self.h), "timer_start")

    def timer_stop(self) -> float:
        ms = C.c_double()
        _check(lib().slimt_b200_timer_stop(self.h, C.byref(ms)), "timer_stop")
        return ms.value

    def profile(self, on: bool):
        _check(lib().slimt_b200_profile_enable(self.h, int(on)), "profile_enable")

    def profile_read(self):
        arr = (KernelStat * 64)()
        n = C.c_size_t()
        _check(lib().slimt_b200_profile_read(self.h, arr, 64, C.byref(n)), "profile_read")
        return [{"name": arr[i].name.decode(), "launches": int(arr[i].launches), "ms": arr[i].ms, "ops": arr[i].ops,
                 "bytes": arr[i].bytes} for i in range(min(n.value, 64))]

    def flush_l2(self, nbytes: int = 256 << 20):
        _check(lib().slimt_b200_flush_l2(self.h, nbytes), "flush_l2")

    def to_device(self, a: np.ndarray) -> int:
        a = np.ascontiguousarray(a)
        p = lib().slimt_b200_dev_alloc(self.h, max(a.nbytes, 16))
        if not p:
            raise RuntimeError(_err())
        _check(lib().slimt_b200_memcpy_h2d(self.h, p, _ptr(a), a.nbytes), "memcpy_h2d")
        return p

    def dev_alloc(self, nbytes: int) -> int:
        p = lib().slimt_b200_dev_alloc(self.h, max(nbytes, 16))
        if not p:
            raise RuntimeError(_err())
        return p

    def from_device(self, p: int, shape, dtype) -> np.ndarray:
        out = np.empty(shape, dtype=dtype)
        _check(lib().slimt_b200_memcpy_d2h(self.h, _ptr(out), p, out.nbytes), "memcpy_d2h")
        return out

    def dev_free(self, p: int):
        lib().slimt_b200_dev_free(self.h, p)

    # qmm::affine / dot / affine_with_select (slimt/QMM.hh:48-63)
    def qmm_affine(self, x: np.ndarray, W: np.ndarray, bias: Optional[np.ndarray], a_quant: float, b_quant: float,
                   indices: Optional[np.ndarray] = None, debug: bool = False):
        x = np.ascontiguousarray(x, dtype=np.float32)
        W = np.ascontiguousarray(W, dtype=np.int8)
        M, K = x.shape
        N = W.shape[0]
        b = None if bias is None else np.ascontiguousarray(bias, dtype=np.float32).reshape(-1)
        idx = None if indices is None else np.ascontiguousarray(indices, dtype=np.uint32)
        nout = N if idx is None else len(idx)
        y = np.empty((M, nout), dtype=np.float32)
        qa = np.empty((M, K), dtype=np.int8) if debug else None
        acc = np.empty((M, nout), dtype=np.int32) if debug else None
        _check(lib().slimt_b200_qmm_affine_debug(self.h, _ptr(x), M, K, _ptr(W), N, _ptr(b), a_quant, b_quant, _ptr(idx),
                                                 0 if idx is None else len(idx), _ptr(y), _ptr(qa), _ptr(acc)),
               "slimt_b200_qmm_affine")
        return (y, qa, acc) if debug else y


class Model:
    def __init__(self, ctx: Context, model_bin: bytes, encoder_layers=6, decoder_layers=2, num_heads=8, eos_id=0, pad_id=0):
        self.ctx = ctx
        self.h = C.c_void_p()
        cfg = ModelConfig(encoder_layers, decoder_layers, 2, num_heads, eos_id, pad_id)
        buf = (C.c_char * len(model_bin)).from_buffer_copy(model_bin)
        _check(lib().slimt_b200_model_create(ctx.h, buf, len(model_bin), C.byref(cfg), C.byref(self.h)),
               "slimt_b200_model_create")
        e, f, v = C.c_int32(), C.c_int32(), C.c_int32()
        lib().slimt_b200_model_dims(self.h, C.byref(e), C.byref(f), C.byref(v))
        self.E, self.F, self.V = e.value, f.value, v.value

    def close(self):
        if self.h:
            lib().slimt_b200_model_destroy(self.h)
            self.h = C.c_void_p()

    def set_max_length(self, n: int):
        """Longest sentence the model accepts, within [1, max_length()[1]] (default 256)."""
        _check(lib().slimt_b200_model_set_max_length(self.h, int(n)), "slimt_b200_model_set_max_length")

    def max_length(self):
        """(current bound, largest bound the model supports)."""
        cur, sup = C.c_int32(), C.c_int32()
        _check(lib().slimt_b200_model_max_length(self.h, C.byref(cur), C.byref(sup)), "slimt_b200_model_max_length")
        return cur.value, sup.value

    def forward(self, tokens: np.ndarray, lengths: np.ndarray, limit_factor: float = 1.5,
                shortlist: Optional[np.ndarray] = None, forced: Optional[np.ndarray] = None,
                want_encoder: bool = False, want_logits: bool = False, want_alignment: bool = False):
        """Model::forward on host buffers. Returns dict(step_tokens [steps,B], steps, target_tokens, ...)."""
        tokens = np.ascontiguousarray(tokens, dtype=np.uint32)
        lengths = np.ascontiguousarray(lengths, dtype=np.uint32)
        B, T = tokens.shape
        max_steps = max(1, int(np.float32(limit_factor) * np.float32(T)))
        sl = None if shortlist is None else np.ascontiguousarray(shortlist, dtype=np.uint32)
        nout = self.V if sl is None else len(sl)
        fo = None if forced is None else np.ascontiguousarray(forced, dtype=np.uint32)
        steps = np.zeros((max(1, max_steps), B), dtype=np.uint32)
        enc = np.empty((B, T, self.E), dtype=np.float32) if want_encoder else None
        logits = np.zeros((max(1, max_steps), B, nout), dtype=np.float32) if want_logits else None
        align = np.zeros((max(1, max_steps), B, T), dtype=np.float32) if want_alignment else None
        io = ForwardIO(_ptr(tokens), _ptr(lengths), B, T, limit_factor, _ptr(sl), 0 if sl is None else len(sl), _ptr(fo),
                       0, _ptr(steps), 0, 0, _ptr(enc), _ptr(logits), _ptr(align))
        _check(lib().slimt_b200_model_forward(self.h, C.byref(io)), "slimt_b200_model_forward")
        n = int(io.steps)
        return {"step_tokens": steps[:n], "steps": n, "target_tokens": int(io.target_tokens), "encoder_out": enc,
                "logits": None if logits is None else logits[:n], "alignment": None if align is None else align[:n]}

    def forward_resident(self, d_tokens: int, d_lengths: int, B: int, T: int, d_steps: int, limit_factor: float = 1.5,
                         d_shortlist: int = 0, n_shortlist: int = 0):
        """Model::forward with inputs/outputs already in HBM (no host<->device copies of the batch)."""
        io = ForwardIO(d_tokens, d_lengths, B, T, limit_factor, d_shortlist or None, n_shortlist, None, 1, d_steps, 0, 0,
                       None, None, None)
        _check(lib().slimt_b200_model_forward(self.h, C.byref(io)), "slimt_b200_model_forward")
        return int(io.steps), int(io.target_tokens)

    def translate_flat(self, tokens: np.ndarray, offsets: np.ndarray, max_words: int, limit_factor: float = 1.5,
                       shortlist_bin: Optional[bytes] = None, out_tokens: Optional[np.ndarray] = None,
                       out_offsets: Optional[np.ndarray] = None, replicas=None, want_alignments: bool = False,
                       shortlist_check: bool = False, shortlist_shared: bool = False):
        """slimt_b200_translate (or _translate_multi over `replicas`, a list of Models) on caller-owned host buffers:
        ragged sentences in (tokens, offsets), ragged targets out (out_tokens, out_offsets).  This is the C-ABI call a
        host integration makes; nothing is repacked."""
        n = len(offsets) - 1
        lens = np.diff(offsets.astype(np.int64))
        max_len = int(lens.max()) if n else 0
        per = max(1, int(np.float32(limit_factor) * np.float32(max_len)))
        if out_offsets is None:
            out_offsets = np.zeros(n + 1, dtype=np.uint64)
        if out_tokens is None:
            out_tokens = np.zeros(max(1, n * per), dtype=np.uint32)
        align = align_offs = None
        if want_alignments:
            align = np.zeros(max(1, per * int(lens.sum())), dtype=np.float32)  # upper bound: every sentence decoded to the limit
            align_offs = np.zeros(n + 1, dtype=np.uint64)
        slbuf = None
        if shortlist_bin is not None:
            slbuf = shortlist_bin if isinstance(shortlist_bin, C.Array) else (C.c_char * len(shortlist_bin)).from_buffer_copy(shortlist_bin)
        io = TranslateIO(_ptr(tokens), _ptr(offsets), n, max_words, limit_factor,
                         C.cast(slbuf, C.c_void_p) if slbuf is not None else None,
                         0 if slbuf is None else len(slbuf), int(shortlist_check), int(shortlist_shared),
                         _ptr(out_tokens), len(out_tokens), _ptr(out_offsets),
                         _ptr(align), 0 if align is None else len(align), _ptr(align_offs), 0, 0, 0.0, 0, 0, 0)
        if replicas is None:
            _check(lib().slimt_b200_translate(self.h, C.byref(io)), "slimt_b200_translate")
        else:
            hs = (C.c_void_p * len(replicas))(*[r.h for r in replicas])
            _check(lib().slimt_b200_translate_multi(hs, len(replicas), C.byref(io)), "slimt_b200_translate_multi")
        stats = {"target_tokens": int(io.target_tokens), "batches": int(io.batches), "device_ms": io.device_ms,
                 "kernel_launches": int(io.kernel_launches), "h2d_bytes": int(io.h2d_bytes),
                 "d2h_bytes": int(io.d2h_bytes)}
        if want_alignments:
            stats["alignments"], stats["align_offsets"] = align, align_offs
        return out_tokens, out_offsets, stats

    def translate(self, sentences, max_words: int, limit_factor: float = 1.5, shortlist_bin: Optional[bytes] = None,
                  replicas=None, want_alignments: bool = False, **kw):
        """exhaust() over one request: Batcher + shortlist + forward per batch, host buffers in and out."""
        offsets = np.zeros(len(sentences) + 1, dtype=np.uint64)
        offsets[1:] = np.cumsum([len(s) for s in sentences])
        tokens = np.concatenate([np.asarray(s, dtype=np.uint32) for s in sentences]) if sentences else np.zeros(0, np.uint32)
        out_tokens, out_offsets, stats = self.translate_flat(tokens, offsets, max_words, limit_factor, shortlist_bin,
                                                             replicas=replicas, want_alignments=want_alignments, **kw)
        outs = [out_tokens[int(out_offsets[i]):int(out_offsets[i + 1])].copy() for i in range(len(sentences))]
        if want_alignments:
            al, ao = stats.pop("alignments"), stats.pop("align_offsets")
            stats["alignments"] = [al[int(ao[i]):int(ao[i + 1])].reshape(len(outs[i]), len(sentences[i])).copy()
                                   for i in range(len(sentences))]
        return outs, stats
