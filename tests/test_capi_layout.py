"""CPU: the ctypes mirrors in slimt_b200/capi.py have the C ABI's layout.  A small C program compiled against
include/slimt_b200.h prints sizeof and every field's offsetof for the two I/O structs; each ctypes field must sit at
the same offset, so a field appended to the header (token_scores, out_scores) cannot drift from its mirror."""
import os
import subprocess

import pytest

from slimt_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STRUCTS = {"slimt_b200_forward_io": capi.ForwardIO, "slimt_b200_translate_io": capi.TranslateIO}


@pytest.fixture(scope="module")
def c_layout(tmp_path_factory):
    tmp = tmp_path_factory.mktemp("layout")
    lines = ['#include <stddef.h>', '#include <stdio.h>', '#include "slimt_b200.h"', "int main(void) {"]
    for cname, py in STRUCTS.items():
        lines.append(f'  printf("{cname} sizeof %zu\\n", sizeof({cname}));')
        for field, _ in py._fields_:
            lines.append(f'  printf("{cname} {field} %zu\\n", offsetof({cname}, {field}));')
    lines += ["  return 0;", "}"]
    src, exe = tmp / "layout.c", tmp / "layout"
    src.write_text("\n".join(lines) + "\n")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split("\n")
    return {(l.split()[0], l.split()[1]): int(l.split()[2]) for l in out if l}


@pytest.mark.parametrize("cname", sorted(STRUCTS))
def test_ctypes_offsets_match_header(c_layout, cname):
    py = STRUCTS[cname]
    for field, _ in py._fields_:
        assert getattr(py, field).offset == c_layout[(cname, field)], field
    assert __import__("ctypes").sizeof(py) == c_layout[(cname, "sizeof")]


def test_new_fields_are_last():
    """Appended, so positional ForwardIO(...) / TranslateIO(...) calls written before them stay valid."""
    assert capi.ForwardIO._fields_[-1][0] == "token_scores"
    assert capi.TranslateIO._fields_[-1][0] == "out_scores"
