#!/usr/bin/env python3
"""TEST INFRASTRUCTURE (BPE_LIB_PATH = the emulator build): BasicTokenizer / RegexTokenizer .train() of the product classes
(kernels on the emulator) against what the UNMODIFIED reference classes did on the same random small texts
(tests/golden/golden_fuzz_train.json, written by tests/golden/make_golden_ref_checks.py) — tie-heavy alphabets, runs of one
character (the (a,a) path), texts that run out of pairs (both must raise ValueError and leave the tokenizer untrained),
both split patterns; merges, vocab, the ids of encode() and the saved .model / .vocab bytes must be identical.

    BPE_LIB_PATH=tests/emu/_build/libb200bpe_emu.so python tests/emu/emu_fuzz_train_ref.py
"""
import hashlib
import json
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import minbpe_b200 as ours  # noqa: E402
from minbpe_b200.tokenizer import GPT2_SPLIT_PATTERN, GPT4_SPLIT_PATTERN  # noqa: E402


def sha(b):
    return hashlib.sha256(b).hexdigest()


def main():
    with open(os.path.join(ROOT, "tests", "golden", "golden_fuzz_train.json"), encoding="utf-8") as f:
        cases = json.load(f)["cases"]
    done = raised = 0
    tmp = tempfile.mkdtemp()
    for it, c in enumerate(cases):
        text, vocab, which = c["text"], c["vocab_size"], c["tokenizer"]
        if which == "basic":
            o = ours.BasicTokenizer()
        else:
            o = ours.RegexTokenizer(GPT4_SPLIT_PATTERN if which == "gpt4" else GPT2_SPLIT_PATTERN)
        err = None
        try:
            o.train(text, vocab)
        except ValueError as ex:
            err = ex
        assert (err is not None) == ("raises" in c), (it, which, vocab, text, err)
        if err is not None:
            raised += 1
            assert not getattr(o, "merges", None) or o.merges == {}, "a failed train() must not leave merges behind"
            continue
        assert list(o.merges.items()) == [((a, b), 256 + i) for i, (a, b) in enumerate(c["merges"])], (it, which, vocab, text)
        want_vocab = {i: bytes([i]) for i in range(256)}
        want_vocab.update({256 + i: bytes.fromhex(h) for i, h in enumerate(c["vocab_hex"])})
        assert o.vocab == want_vocab
        probe = text[: 300] + " ab aab" + text[-50:]
        ids = o.encode(probe)
        assert (len(ids), sha(np.asarray(ids, dtype="<i4").tobytes())) == (c["probe_n_ids"], c["probe_ids_sha256"]), (it, which, probe)
        assert o.decode(ids) == probe
        o.save(os.path.join(tmp, "o"))
        for ext in ("model", "vocab"):
            assert sha(open(os.path.join(tmp, "o." + ext), "rb").read()) == c[ext + "_sha256"], (it, ext)
        done += 1
    print(f"emu fuzz train ok: {done} trained identically, {raised} ran out of pairs on both sides, of {len(cases)}")
    return 0


if __name__ == "__main__":
    sys.exit(main())
