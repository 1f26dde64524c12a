"""CPU: the ctypes mirror of slimt_b200_beam has the C header's layout (sizeof and every field's offsetof, from a small C
program compiled against include/slimt_b200.h), and the beam entry point is exported."""
import ctypes
import os
import subprocess

from slimt_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_beam_offsets_match_header(tmp_path):
    name, py = "slimt_b200_beam", capi.Beam
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


def test_beam_entry_point_exported():
    assert "slimt_b200_translate_beam" in capi.EXPORTS
    getattr(capi.lib(), "slimt_b200_translate_beam")
