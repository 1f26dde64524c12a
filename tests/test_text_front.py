"""The text front half (include/slimt_b200_text.hh; SURVEY.md section 8 f4): sentencepiece Vocabulary, sentence
splitter, TextProcessor, AnnotatedText, Response / combine.

1. Every command of tests/golden/text/golden.json -- answered by the UNMODIFIED reference (its Vocabulary.cc,
   TextProcessor.cc, Splitter.cc, Regex.cc, Annotation.cc, Response.cc, Request.cc with the vendored sentencepiece
   0.2.00, compiled in place; tests/golden/make_text_golden.py) -- is replayed through the product's host code behind the
   same driver (tests/cpp/text_front_driver.cc) and must be answered byte for byte the same.
2. Vocabulary::encode / decode against the sentencepiece wheel's stored answers on seeded random strings.
3. Where the reference sources exist (this container), the freshly built reference driver and the product driver are
   compared live on further random inputs."""
import hashlib
import json
import os
import random
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "tests", "cpp", "text_front_test")
GOLD = os.path.join(ROOT, "tests", "golden", "text")
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "text_ref")


@pytest.fixture(scope="module")
def driver():
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "slimt_b200", "csrc"), "text_test"])
    assert os.path.exists(BIN)
    return BIN


def _run(binary, commands):
    r = subprocess.run([binary], input="\n".join(commands) + "\n", capture_output=True, text=True, cwd=ROOT, check=True)
    out = r.stdout.split("\n")[:-1]
    assert len(out) == len(commands), (len(out), len(commands), r.stderr[-500:])
    return out


def _golden():
    return json.load(open(os.path.join(GOLD, "golden.json")))["pairs"]


def test_golden_answers_of_the_reference(driver):
    pairs = _golden()
    assert len(pairs) > 500
    kinds = {c.split()[0] for c, _ in pairs}
    assert kinds == {"vocab", "encode", "decode", "split", "process", "recode", "respond", "pivot"}
    got = _run(driver, [c for c, _ in pairs])
    bad = [(c, want, have) for (c, want), have in zip(pairs, got) if want != have]
    assert not bad, f"{len(bad)} of {len(pairs)} answers differ; first: {bad[0][0][:120]!r}\n want {bad[0][1][:300]}\n have {bad[0][2][:300]}"


def _hx(s):
    b = s if isinstance(s, bytes) else s.encode("utf-8")
    return b.hex() if b else "-"


ALPHABET = list("abcdefghijklmnopqrstuvwxyzäöüéèñç") + list("αβγδεζηθ") + list("абвгдежз") + list("日本語中文翻訳") + \
    [" ", " ", " ", "  ", ".", ",", "!", "?", "\t", "\n", "<br>", "@@", "😀", "Ａ", "ﬁ", "①", "é", " ", "　", "▁", "0", "7", "42"]


def _random_text(rng, lo=0, hi=40):
    return "".join(rng.choice(ALPHABET) for _ in range(rng.randint(lo, hi)))


def vocabulary_commands(model, pieces):
    """Seeded random strings (malformed UTF-8 included) to encode and id lists to decode, as driver commands."""
    rng = random.Random(31337 if model.startswith("spm_u") else 271828)
    texts = [_random_text(rng).encode("utf-8") for _ in range(400)]
    for _ in range(60):  # random byte damage
        b = bytearray(_random_text(rng, 5, 30).encode("utf-8"))
        for _ in range(rng.randint(1, 3)):
            b[rng.randrange(len(b))] = rng.randrange(256)
        texts.append(bytes(b))
    id_lists = [[rng.randrange(pieces) for _ in range(rng.randint(0, 25))] for _ in range(300)]
    cmds = [f"vocab {os.path.join('tests', 'golden', 'text', model)}"] + [f"encode {_hx(t)}" for t in texts] + \
        ["decode " + " ".join(map(str, ids)) for ids in id_lists]
    return texts, id_lists, cmds


@pytest.mark.parametrize("model", ["spm_unigram.model", "spm_bytes.model"])
def test_vocabulary_against_the_sentencepiece_wheel(driver, model):
    """Encode: ids and the byte range of every piece (SentencePieceText.pieces[].begin / end); Decode: text and ranges.
    Includes malformed UTF-8, where only the ids are compared (offsets are pinned by the reference goldens).  The
    wheel's answers are stored in tests/golden/text/wheel.json (tests/golden/make_wheel_golden.py)."""
    g = json.load(open(os.path.join(GOLD, "wheel.json")))["vocabulary"][model]
    _, _, cmds = vocabulary_commands(model, g["pieces"])
    assert hashlib.sha256("\n".join(cmds).encode("utf-8")).hexdigest() == g["commands_sha256"], "inputs drifted"
    got = _run(driver, cmds)[1:]
    assert len(got) == len(g["answers"])
    bad = [(c, want, have) for c, want, have in zip(cmds[1:], g["answers"], got)
           if (have if " |" in want else have.split(" |")[0]) != want]
    assert not bad, f"{len(bad)} of {len(got)} answers differ; first: {bad[0][0][:120]!r}\n want {bad[0][1][:300]}\n have {bad[0][2][:300]}"


@pytest.mark.skipif(not os.path.isdir("/root/reference/slimt"), reason="the reference sources only exist in the build container")
def test_live_against_the_reference_build(driver):
    subprocess.check_call(["make", "-s", "-j8", "-C", os.path.join(ROOT, "oracle"), "text_ref"])
    rng = random.Random(8086)
    words = ["Word", "word", "Xy", "it", "12", "3", ".", "!", "?", "...", " ", " ", " ", "  ", "\n", "\n\n", "\"", ")", "]", "[", "Dr", "No",
             "。", "日本", "é", "Ä", "’", "[1]", ",", "а", "Б", "α", "Ω", "\r\n", "։", "？", "e.g", "U.S"]
    prefixes = _hx("Dr\nNo #NUMERIC_ONLY#\ne.g\nU.S\n")
    cmds = ["vocab tests/golden/text/spm_unigram.model"]
    for _ in range(1500):
        text = "".join(rng.choice(words) for _ in range(rng.randint(0, 40)))
        mode = rng.choice(["sentence", "paragraph", "wrapped_text"])
        cmds.append(f"split {mode} {rng.choice(['-', prefixes])} {_hx(text)}")
        cmds.append(f"process {mode} {rng.choice([2, 3, 7, 128])} {_hx(text)}")
        cmds.append(f"recode {mode} 128 {_hx(text)}")
        cmds.append(f"encode {_hx(_random_text(rng))}")
    assert _run(driver, cmds) == _run(REF_BIN, cmds)


def test_damaged_vocabulary_files_are_refused_not_crashed_on(driver):
    """Truncated, bit-flipped and spliced sentencepiece files (incl. damage inside the precompiled character map and its
    double-array trie): the loader either throws or yields a vocabulary that still encodes and decodes; the process
    survives (clean under -fsanitize=address,undefined as well)."""
    out = _run(driver, ["loadfuzz tests/golden/text/spm_unigram.model 7 300", "loadfuzz tests/golden/text/spm_bytes.model 9 300"])
    for line in out:
        got = dict(kv.split("=") for kv in line.split()[1:])
        assert int(got["loaded"]) + int(got["refused"]) == 300 and int(got["refused"]) > 100


@pytest.mark.skipif(not os.path.isdir("/root/reference/slimt"), reason="the reference sources only exist in the build container")
def test_live_against_the_reference_build_on_real_text(driver):
    """Half a megabyte of real English prose with code, lists, quotes, abbreviations and numbers (the Python documentation
    topics shipped with the interpreter) through the splitter in all three modes and through TextProcessor::process."""
    topics = pytest.importorskip("pydoc_data.topics")
    subprocess.check_call(["make", "-s", "-j8", "-C", os.path.join(ROOT, "oracle"), "text_ref"])
    text = "\n\n".join(topics.topics.values())
    chunks, cur = [], ""
    for para in text.split("\n\n"):
        cur += para + "\n\n"
        if len(cur) > 3000:
            chunks.append(cur)
            cur = ""
    cmds = ["vocab tests/golden/text/spm_unigram.model"]
    for c in chunks:
        for mode in ("wrapped_text", "paragraph", "sentence"):
            cmds.append(f"split {mode} - {_hx(c)}")
        cmds.append(f"process wrapped_text 64 {_hx(c)}")
    assert len(cmds) > 400
    assert _run(driver, cmds) == _run(REF_BIN, cmds)
