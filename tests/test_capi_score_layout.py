"""CPU: the ctypes mirror of slimt_b200_score_io has the C header's layout (sizeof and every field's offsetof, from a
small C program compiled against include/slimt_b200.h), slimt_b200_score is exported, and the request checks that need
no model -- offsets that decrease, an output capacity too small -- fail before anything else is looked at."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from slimt_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_score_io_offsets_match_header(tmp_path):
    name, py = "slimt_b200_score_io", capi.ScoreIO
    lines = ['#include <stddef.h>', '#include <stdio.h>', '#include "slimt_b200.h"', "int main(void) {",
             f'  printf("sizeof %zu\\n", sizeof({name}));']
    lines += [f'  printf("{f} %zu\\n", offsetof({name}, {f}));' for f, _ in py._fields_]
    lines += ["  return 0;", "}"]
    src, exe = tmp_path / "layout.c", tmp_path / "layout"
    src.write_text("\n".join(lines) + "\n")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split("\n") if l)
    for f, _ in py._fields_:
        assert getattr(py, f).offset == int(got[f]), f
    assert ctypes.sizeof(py) == int(got["sizeof"])


def test_score_exported():
    assert "slimt_b200_score" in capi.EXPORTS
    capi.lib().slimt_b200_score


def _request():
    tokens = np.array([5, 6, 0, 7, 0], dtype=np.uint32)
    offsets = np.array([0, 3, 5], dtype=np.uint64)
    targets = np.array([9, 0, 8, 0], dtype=np.uint32)
    target_offsets = np.array([0, 2, 4], dtype=np.uint64)
    return tokens, offsets, targets, target_offsets


@pytest.mark.parametrize("bad,msg", [("offsets", "non-decreasing"), ("target_offsets", "non-decreasing"),
                                     ("capacity", "capacity too small"), ("align_capacity", "capacity too small"),
                                     ("replicas", "no model replica")])
def test_score_rejects_malformed_request_without_a_device(bad, msg):
    tokens, offsets, targets, target_offsets = _request()
    kw = {}
    if bad == "offsets":
        offsets = np.array([0, 3, 2], dtype=np.uint64)
    elif bad == "target_offsets":
        target_offsets = np.array([0, 2, 1], dtype=np.uint64)
    elif bad == "capacity":
        kw["out_capacity"] = 3
    elif bad == "align_capacity":
        kw["want_alignments"], kw["align_capacity"] = True, 9
    with pytest.raises(RuntimeError, match=msg):
        capi.score_flat([], tokens, offsets, targets, target_offsets, max_words=64, **kw)
