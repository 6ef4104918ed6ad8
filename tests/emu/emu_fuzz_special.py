#!/usr/bin/env python3
"""TEST INFRASTRUCTURE (BPE_LIB_PATH = the emulator build): RegexTokenizer.encode(text, allowed_special=...) with the
special tokens found, the parts split and everything encoded on the device (k_special.cuh, split_logic.h WITH_B,
k_encode2.cuh) against the ids the UNMODIFIED reference class returned for the same random texts
(tests/golden/golden_fuzz_special.json, written by tests/golden/make_golden_ref_checks.py): specials that are prefixes of
one another, adjacent and overlapping occurrences, specials at either end of the text, white space / letters / digits /
apostrophes on both sides (the split of a part must behave as on a text of its own), both split patterns, subsets as
`allowed_special`, several pieces per call.

    BPE_LIB_PATH=tests/emu/_build/libb200bpe_emu.so python tests/emu/emu_fuzz_special.py
"""
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from minbpe_b200 import RegexTokenizer  # noqa: E402
from minbpe_b200 import engine as E  # noqa: E402
from minbpe_b200.tokenizer import GPT2_SPLIT_PATTERN, GPT4_SPLIT_PATTERN  # noqa: E402


def ids_sha(ids):
    return hashlib.sha256(np.asarray(ids, dtype="<i4").tobytes()).hexdigest()


def main():
    with open(os.path.join(ROOT, "tests", "golden", "golden_fuzz_special.json"), encoding="utf-8") as f:
        g = json.load(f)
    toks = {}
    for name, pat in (("gpt4", GPT4_SPLIT_PATTERN), ("gpt2", GPT2_SPLIT_PATTERN)):
        o = RegexTokenizer(pat)
        o.merges = {(a, b): 256 + i for i, (a, b) in enumerate(g["merges"][name])}   # the reference's trained merges
        o.vocab = o._build_vocab()
        o.DEVICE_SPLIT_MIN_BYTES = 0          # every text takes the device path, however short
        toks[name] = o
    n_dev = 0
    for it, c in enumerate(g["cases"]):
        o, text = toks[c["pattern"]], c["text"]
        o.register_special_tokens(c["special"])
        allowed = c["allowed"] if c["allowed"] == "all" else set(c["allowed"])
        o.engine.set_option(E.OPT_SPLIT_PIECE, c["piece"])
        try:
            try:
                got = o.encode(text, allowed_special=allowed)
            except E.EngineError as ex:       # a tiny piece size may find no letter+space cut: a clean error, not a wrong answer
                assert "cut point" in str(ex), ex
                continue
        finally:
            o.engine.set_option(E.OPT_SPLIT_PIECE, 0)
        assert (len(got), ids_sha(got)) == (c["n_ids"], c["ids_sha256"]), (it, c["pattern"], c["special"], c["allowed"], text)
        assert o.decode(got) == text
        n_dev += 1
    print(f"emu fuzz special ok: {n_dev} of {len(g['cases'])} rounds compared with the reference class")
    return 0


if __name__ == "__main__":
    sys.exit(main())
