"""CPU: the top-k entry points are exported, the "top_k" key of the sampling dict reaches them (through a stand-in for
the library), and the C++ services program for Options::top_k builds."""
import ctypes as C
import os
import subprocess

import numpy as np

from slimt_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_topk_entry_points_exported():
    lib = capi.lib()
    for name in ("slimt_b200_model_forward_topk", "slimt_b200_translate_topk"):
        assert name in capi.EXPORTS
        getattr(lib, name)


class _Recorder:
    """Stands in for the library: records which entry point was called with which top_k and sampling struct."""

    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        def call(*args):
            self.calls.append((name, args))
            return 0
        return call


def _model(monkeypatch):
    rec = _Recorder()
    monkeypatch.setattr(capi, "lib", lambda: rec)
    m = object.__new__(capi.Model)
    m.h, m.V, m.E = C.c_void_p(1), 64, 32
    return m, rec


def test_top_k_key_reaches_the_forward_call(monkeypatch):
    m, rec = _model(monkeypatch)
    tokens, lengths = np.ones((2, 3), dtype=np.uint32), np.array([3, 2], dtype=np.uint32)
    m.forward(tokens, lengths, sampling={"temperature": 0.5, "seed": 9, "top_k": 17})
    name, args = rec.calls[-1]
    assert name == "slimt_b200_model_forward_topk" and args[-1] == 17
    sp = args[2]._obj
    assert sp.temperature == 0.5 and sp.seed == 9
    m.forward(tokens, lengths, sampling={"temperature": 0.5, "seed": 9, "top_k": 0})
    assert rec.calls[-1][0] == "slimt_b200_model_forward_topk" and rec.calls[-1][1][-1] == 0
    m.forward(tokens, lengths, sampling={"temperature": 0.5})
    assert rec.calls[-1][0] == "slimt_b200_model_forward_sampled"
    m.forward_resident(1, 2, 2, 3, 4, sampling={"temperature": 1.0, "keys": 1234, "top_k": 5})
    name, args = rec.calls[-1]
    assert name == "slimt_b200_model_forward_topk" and args[-1] == 5 and args[2]._obj.keys == 1234


def test_top_k_key_reaches_the_translate_call(monkeypatch):
    m, rec = _model(monkeypatch)
    sents = [np.array([5, 6, 0], dtype=np.uint32), np.array([7, 0], dtype=np.uint32)]
    m.translate(sents, max_words=64, sampling={"temperature": 2.0, "seed": 1, "top_k": 256})
    name, args = rec.calls[-1]
    assert name == "slimt_b200_translate_topk" and args[1] == 1 and args[-1] == 256
    m.translate(sents, max_words=64, sampling={"temperature": 2.0})
    assert rec.calls[-1][0] == "slimt_b200_translate_sampled"


def test_topk_program_builds():
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "slimt_b200", "csrc"), "host_topk"])
    assert os.path.exists(os.path.join(ROOT, "tests", "cpp", "host_topk_test"))
