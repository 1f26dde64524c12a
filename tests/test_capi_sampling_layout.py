"""CPU: the ctypes mirror of slimt_b200_sampling has the C header's layout (sizeof and every field's offsetof, from a
small C program compiled against include/slimt_b200.h), and the sampled entry points are exported."""
import ctypes
import os
import subprocess

from slimt_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_sampling_offsets_match_header(tmp_path):
    name, py = "slimt_b200_sampling", capi.Sampling
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


def test_sampled_entry_points_exported():
    lib = capi.lib()
    for name in ("slimt_b200_model_forward_sampled", "slimt_b200_translate_sampled"):
        assert name in capi.EXPORTS
        getattr(lib, name)


def test_sampling_struct_from_dict():
    import numpy as np
    sp, keys = capi._sampling({"temperature": 0.5, "seed": 2**64 - 1, "keys": [3, 2**63]})
    assert sp.temperature == 0.5 and sp.seed == 2**64 - 1
    assert keys.dtype == np.uint64 and sp.keys == keys.ctypes.data
    sp, keys = capi._sampling({"temperature": 2.0}, device_keys=True)
    assert sp.keys is None and sp.seed == 0
    assert capi._sampling(None) == (None, None)
