"""CPU: the sampling generator (slimt_b200/csrc/sample_rng.cuh), compiled for the host, reproduces Random123's
Philox4x32-10 known answers, equals a numpy restatement of the uniform-number construction, and its u is uniform."""
import os
import subprocess

import numpy as np
import pytest
from scipy import stats

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# Random123 kat_vectors: philox4x32 10 rounds, counter / key / output
KAT = [
    ("00000000 00000000 00000000 00000000", "00000000 00000000", "6627e8d5 e169c58d bc57ac4c 9b00dbd8"),
    ("ffffffff ffffffff ffffffff ffffffff", "ffffffff ffffffff", "408f276d 41c83b0e a20bc7c6 6d5451fd"),
    ("243f6a88 85a308d3 13198a2e 03707344", "a4093822 299f31d0", "d16cfe09 94fdcceb 5001e420 24126ea1"),
]


@pytest.fixture(scope="module")
def rng_bin(tmp_path_factory):
    exe = tmp_path_factory.mktemp("rng") / "sample_rng_test"
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "slimt_b200", "csrc"),
                           os.path.join(ROOT, "tests", "cpp", "sample_rng_test.cc"), "-o", str(exe)])
    return str(exe)


def _run(exe, lines):
    r = subprocess.run([exe], input="\n".join(lines) + "\n", capture_output=True, text=True, check=True)
    return r.stdout.split()


def philox_np(c, k):
    """Philox4x32-10 over arrays: c = 4 uint32 arrays, k = 2 uint32 arrays (numpy restatement)."""
    c0, c1, c2, c3 = (np.asarray(x, dtype=np.uint64) for x in c)
    k0, k1 = (np.asarray(x, dtype=np.uint64) for x in k)
    m32 = np.uint64(0xFFFFFFFF)
    for r in range(10):
        if r:
            k0, k1 = (k0 + np.uint64(0x9E3779B9)) & m32, (k1 + np.uint64(0xBB67AE85)) & m32
        p0, p1 = np.uint64(0xD2511F53) * c0, np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & m32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & m32
    return c0, c1, c2, c3


def uniform_np(seed, key, step):
    """u * 2^53 of include/slimt_b200.h's definition, as uint64."""
    seed, key = np.asarray(seed, dtype=np.uint64), np.asarray(key, dtype=np.uint64)
    m32, s32 = np.uint64(0xFFFFFFFF), np.uint64(32)
    x0, x1, _, _ = philox_np((np.asarray(step, dtype=np.uint64), key & m32, key >> s32, np.zeros_like(key)),
                             (seed & m32, seed >> s32))
    return ((x0 << s32) | x1) >> np.uint64(11)


def test_known_answers(rng_bin):
    out = _run(rng_bin, [f"philox {c} {k}" for c, k, _ in KAT])
    assert [" ".join(out[4 * i:4 * i + 4]) for i in range(len(KAT))] == [o for _, _, o in KAT]


def test_numpy_restatement_matches():
    for c, k, o in KAT:
        got = philox_np([int(x, 16) for x in c.split()], [int(x, 16) for x in k.split()])
        assert " ".join(f"{int(x):08x}" for x in got) == o


def test_host_build_matches_numpy_and_is_uniform(rng_bin):
    rs = np.random.default_rng(2026)
    n = 100_000
    seed = rs.integers(0, 2**64, n, dtype=np.uint64)
    key = rs.integers(0, 2**64, n, dtype=np.uint64)
    step = rs.integers(0, 1024, n, dtype=np.uint64)
    seed[:100], key[:100], step[:100] = 0, np.arange(100, dtype=np.uint64), 0  # the defaults: seed 0, key = index
    got = np.array([int(x) for x in _run(rng_bin, [f"u {s} {k} {t}" for s, k, t in zip(seed, key, step)])],
                   dtype=np.uint64)
    want = uniform_np(seed, key, step)
    assert np.array_equal(got, want)
    u = want.astype(np.float64) * 2.0**-53
    assert u.min() >= 0.0 and u.max() < 1.0
    assert stats.kstest(u, "uniform").pvalue > 1e-4
