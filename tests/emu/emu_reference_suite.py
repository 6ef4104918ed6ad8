#!/usr/bin/env python3
"""TEST INFRASTRUCTURE (BPE_LIB_PATH = the emulator build): the checks of the reference's own test file
(karpathy/minbpe tests/test_tokenizer.py: encode/decode identity on its test strings, the Wikipedia example, train + save +
load with and without special tokens) run on the product classes, each also compared with what the UNMODIFIED reference
returned (tests/golden/golden_ref_suite.json, written by tests/golden/make_golden_ref_checks.py).  Its GPT4Tokenizer
tests need tiktoken's cl100k_base, a download, and are not part of this.

    BPE_LIB_PATH=tests/emu/_build/libb200bpe_emu.so python tests/emu/emu_reference_suite.py
"""
import hashlib
import json
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
GOLDEN = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, ROOT)
from minbpe_b200 import BasicTokenizer, RegexTokenizer  # noqa: E402


def sha(b):
    return hashlib.sha256(b).hexdigest()


def read(name):
    with open(os.path.join(GOLDEN, name), encoding="utf-8") as f:
        return f.read()


def main():
    g = json.loads(read("golden_ref_suite.json"))
    passed = 0
    for name, cls in (("basic", BasicTokenizer), ("regex", RegexTokenizer)):
        # encode/decode identity of untrained tokenizers
        for s, want in zip(g["test_strings"], g["encode"][name]):
            text = read(s) if s.endswith(".txt") else s
            tok = cls()
            ids = tok.encode(text)
            assert (len(ids), sha(np.asarray(ids, dtype="<i4").tobytes())) == (want["n_ids"], want["ids_sha256"]), (name, s)
            assert tok.decode(ids) == text, (name, s)
            passed += 1
        # Wikipedia example: 3 merges on "aaabdaaabac" give XdXac = [258, 100, 258, 97, 99]
        want = g["wikipedia"][name]
        tok = cls()
        tok.train("aaabdaaabac", 256 + 3)
        assert [list(p) for p in tok.merges] == want["merges"], name
        assert tok.encode("aaabdaaabac") == want["ids"] == [258, 100, 258, 97, 99], name
        assert tok.decode(tok.encode("aaabdaaabac")) == "aaabdaaabac"
        passed += 1
    # train 64 merges on the llama text, register special tokens, save, load into a fresh tokenizer
    text = read("llama_text.txt")
    with tempfile.TemporaryDirectory() as d:
        prefix = os.path.join(d, "tok")
        for want in g["save_load"]:
            tok = RegexTokenizer()
            tok.train(text, 256 + 64)
            tok.register_special_tokens(want["special_tokens"])
            assert [list(p) for p in tok.merges] == want["merges"]
            assert tok.decode(tok.encode(text, "all")) == text
            ids = tok.encode(text, "all")
            assert ids == want["ids"], len(want["special_tokens"])
            tok.save(prefix)
            for ext in ("model", "vocab"):
                assert sha(open(f"{prefix}.{ext}", "rb").read()) == want[ext + "_sha256"], ext
            tok = RegexTokenizer()
            tok.load(prefix + ".model")
            assert tok.decode(ids) == text
            assert tok.decode(tok.encode(text, "all")) == text
            assert tok.encode(text, "all") == ids
            passed += 1
    print(f"reference suite ok: {passed} passed")
    return 0


if __name__ == "__main__":
    sys.exit(main())
