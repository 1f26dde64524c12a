"""Stores the sentencepiece wheel's answers to the vocabulary commands of tests/test_text_front.py
(test_vocabulary_against_the_sentencepiece_wheel) in tests/golden/text/wheel.json, so that the test needs no wheel.

    python tests/golden/make_wheel_golden.py

Encode answers carry the ids and the byte range of every piece (the wheel reports code points, its
ConvertToUnicodeAlignment; the C++ API bytes); for malformed UTF-8 only the ids are stored.  Decode answers carry the text
and the byte ranges of the pieces.
"""
import hashlib
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import sentencepiece as spm  # noqa: E402

from test_text_front import _hx, vocabulary_commands  # noqa: E402


def byte_offsets(text):
    at = [0]
    for ch in text:
        at.append(at[-1] + len(ch.encode("utf-8")))
    return at


def answers(sp, texts, id_lists):
    out = []
    for t in texts:
        try:
            s = t.decode("utf-8")
        except UnicodeDecodeError:
            out.append("ids" + "".join(f" {i}" for i in sp.encode(t, out_type=int)))
            continue
        proto = sp.encode(s, out_type="immutable_proto")
        at = byte_offsets(s)
        out.append("ids" + "".join(f" {p.id}" for p in proto.pieces) + " |" + "".join(f" {at[p.begin]}:{at[p.end]}" for p in proto.pieces))
    for ids in id_lists:
        if not ids:
            out.append("text - |")
            continue
        proto = sp.decode_ids_as_immutable_proto(ids)
        at = byte_offsets(proto.text)
        out.append("text " + _hx(proto.text) + " |" + "".join(f" {at[p.begin]}:{at[p.end]}" for p in proto.pieces))
    return out


def main():
    vocab = {}
    for model in ("spm_unigram.model", "spm_bytes.model"):
        sp = spm.SentencePieceProcessor(model_file=os.path.join(HERE, "text", model))
        texts, id_lists, cmds = vocabulary_commands(model, sp.get_piece_size())
        vocab[model] = {"pieces": sp.get_piece_size(),
                        "commands_sha256": hashlib.sha256("\n".join(cmds).encode("utf-8")).hexdigest(),
                        "answers": answers(sp, texts, id_lists)}
    with open(os.path.join(HERE, "text", "wheel.json"), "w") as f:
        json.dump({"generator": "tests/golden/make_wheel_golden.py", "sentencepiece": spm.__version__, "vocabulary": vocab},
                  f, indent=0, ensure_ascii=True)
        f.write("\n")


if __name__ == "__main__":
    main()
