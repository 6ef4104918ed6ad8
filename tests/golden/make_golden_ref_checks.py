#!/usr/bin/env python3
"""
Golden vectors for the checks that compare minbpe_b200 with the UNMODIFIED reference (karpathy/minbpe @1acefe8) class by
class, so that those checks run without a copy of the reference:

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden_ref_checks.py <karpathy/minbpe checkout>

Outputs (all committed):
  golden_ref_suite.json     what the reference's own tests/test_tokenizer.py checks, with the reference's answers: ids of
                            encode() on its test strings, the Wikipedia example, train + save + load on its llama text
                            with and without special tokens (the GPT4Tokenizer tests need tiktoken's cl100k_base, a
                            download, and are left out)
  golden_fuzz_special.json  random texts and special-token sets (seed 5, 100 rounds) with the ids the reference's
                            RegexTokenizer.encode(text, allowed_special) returns                -> tests/emu/emu_fuzz_special.py
  golden_fuzz_train.json    random small texts (seed 5, 100 rounds) with the reference's train() result: merges, vocab,
                            ids of encode() on a probe, sha256 of the saved files, or that it ran out of pairs
                                                                                               -> tests/emu/emu_fuzz_train_ref.py
The texts and the random cases are data of this project (the strings of the reference's test file are in
llama_text.txt / specials_string.txt and below); nothing here is imported by the product.
"""
import hashlib
import json
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.dont_write_bytecode = True
sys.path.insert(0, ROOT)

from minbpe_b200.tokenizer import GPT2_SPLIT_PATTERN, GPT4_SPLIT_PATTERN  # noqa: E402

PATTERNS = {"gpt4": GPT4_SPLIT_PATTERN, "gpt2": GPT2_SPLIT_PATTERN}

# the strings the reference's test file encodes; "taylorswift.txt" stands for the contents of that file
TEST_STRINGS = ["", "?", "hello world!!!? (안녕하세요!) lol123 😉", "taylorswift.txt"]
SPECIALS = {"<|endoftext|>": 100257, "<|fim_prefix|>": 100258, "<|fim_middle|>": 100259, "<|fim_suffix|>": 100260,
            "<|endofprompt|>": 100276}


def sha(b):
    return hashlib.sha256(b).hexdigest()


def ids_sha(ids):
    return sha(np.asarray(ids, dtype="<i4").tobytes())


def read(name):
    with open(os.path.join(HERE, name), encoding="utf-8") as f:
        return f.read()


def saved(tok):
    """sha256 of the .model and .vocab files tok.save() writes."""
    with tempfile.TemporaryDirectory() as d:
        tok.save(os.path.join(d, "m"))
        return {ext + "_sha256": sha(open(os.path.join(d, "m." + ext), "rb").read()) for ext in ("model", "vocab")}


def ref_suite(ref):
    out = {"test_strings": TEST_STRINGS, "encode": {}, "wikipedia": {}, "save_load": []}
    for name, cls in (("basic", ref.BasicTokenizer), ("regex", ref.RegexTokenizer)):
        rows = []
        for s in TEST_STRINGS:
            text = read(s) if s.endswith(".txt") else s
            ids = cls().encode(text)
            rows.append({"n_ids": len(ids), "ids_sha256": ids_sha(ids)})
        out["encode"][name] = rows
        tok = cls()
        tok.train("aaabdaaabac", 256 + 3)
        out["wikipedia"][name] = {"merges": [list(p) for p in tok.merges], "ids": tok.encode("aaabdaaabac")}
    text = read("llama_text.txt")
    for specials in ({}, SPECIALS):
        tok = ref.RegexTokenizer()
        tok.train(text, 256 + 64)
        tok.register_special_tokens(specials)
        ids = tok.encode(text, "all")
        assert tok.decode(ids) == text
        out["save_load"].append({"special_tokens": specials, "merges": [list(p) for p in tok.merges], "ids": ids, **saved(tok)})
    return out


# ---- special-token front end: random texts and special sets ------------------------------------------------------------
POOL = ["<|endoftext|>", "<|end|>", "<|endof", "<|a|>", "<|a|><|b|>", "<|b|>", "<s>", "</s>", "<s", "[SEP]", "[S", " <pad>", "<|é|>", "'s<", "12", "\n\n<|x|>"]
FILL = list("abcde  é1!'\n\t") + ["日", " the", "'ll", "  ", "\r\n", "42"]


def random_case(rng):
    k = int(rng.integers(1, 6))
    toks = [str(x) for x in rng.choice(POOL, size=k, replace=False)]
    special = {t: 1000 + i for i, t in enumerate(toks)}
    parts = []
    for _ in range(int(rng.integers(1, 60))):
        r = rng.random()
        if r < 0.35:
            parts.append(str(rng.choice(toks)))
        elif r < 0.45:
            t = str(rng.choice(toks))
            parts.append(t[: int(rng.integers(1, len(t) + 1))])          # a truncated special: must stay ordinary text
        else:
            parts.append("".join(str(x) for x in rng.choice(FILL, size=int(rng.integers(1, 12)))))
    return special, "".join(parts)


def fuzz_special(ref, rounds=100, seed=5):
    """Specials that are prefixes of one another, adjacent and overlapping occurrences, specials at either end of the text,
    white space / letters / digits / apostrophes on both sides, both split patterns, subsets as `allowed_special`; `piece` is
    the device split piece size the check uses for that round (0 = whole text)."""
    rng = np.random.default_rng(seed)
    train_text = read("taylorswift.txt")[:60000]
    toks, merges = {}, {}
    for name, pat in PATTERNS.items():
        r = ref.RegexTokenizer(pat)
        r.train(train_text[:20000], 256 + 120)
        toks[name], merges[name] = r, [list(p) for p in r.merges]
    cases = []
    for _ in range(rounds):
        special, text = random_case(rng)
        if rng.random() < 0.2:
            text = text + " " + train_text[: int(rng.integers(100, 5000))] + text
        pat = "gpt4" if rng.random() < 0.6 else "gpt2"
        r = toks[pat]
        r.register_special_tokens(special)
        allowed = "all" if rng.random() < 0.7 else set(list(special)[: int(rng.integers(0, len(special) + 1))])
        piece = int(rng.choice([0, 0, 0, 4096]))
        ids = r.encode(text, allowed_special=allowed)
        assert r.decode(ids) == text
        cases.append({"pattern": pat, "special": special, "allowed": allowed if allowed == "all" else [t for t in special if t in allowed],
                      "piece": piece, "text": text, "n_ids": len(ids), "ids_sha256": ids_sha(ids)})
    return {"train": {"text_chars": 20000, "vocab_size": 256 + 120}, "merges": merges, "cases": cases}


# ---- train(): random small texts ---------------------------------------------------------------------------------------
def random_text(rng):
    kind = rng.random()
    if kind < 0.3:
        alpha = list("ab")                                   # ties everywhere, long runs
    elif kind < 0.6:
        alpha = list("abc de'1\n")
    else:
        alpha = list("the quick brown fox é日 12 's 'll\t") + ["aaaa", "  ", "zzzzzz"]
    n = int(rng.choice([1, 2, 3, 5, 12, 40, 200, 1500]))
    return "".join(str(x) for x in rng.choice(alpha, size=n))


def probe_text(text):
    return text[: 300] + " ab aab" + text[-50:]


def fuzz_train(ref, rounds=100, seed=5):
    """Tie-heavy alphabets, runs of one character (the (a,a) path), texts that run out of pairs (the reference raises
    ValueError), BasicTokenizer and RegexTokenizer with both split patterns."""
    rng = np.random.default_rng(seed)
    cases = []
    for _ in range(rounds):
        text = random_text(rng)
        vocab = 256 + int(rng.choice([0, 1, 2, 5, 20, 60]))
        which = ("basic", "gpt4", "gpt2")[int(rng.integers(0, 3))]
        r = ref.BasicTokenizer() if which == "basic" else ref.RegexTokenizer(PATTERNS[which])
        rec = {"tokenizer": which, "vocab_size": vocab, "text": text}
        try:
            r.train(text, vocab)
        except ValueError:
            rec["raises"] = "ValueError"
            cases.append(rec)
            continue
        assert list(r.merges.values()) == list(range(256, 256 + len(r.merges)))
        assert all(r.vocab[i] == bytes([i]) for i in range(256)) and len(r.vocab) == 256 + len(r.merges)
        rec["merges"] = [list(p) for p in r.merges]
        rec["vocab_hex"] = [r.vocab[256 + i].hex() for i in range(len(r.merges))]
        ids = r.encode(probe_text(text))
        rec["probe_n_ids"], rec["probe_ids_sha256"] = len(ids), ids_sha(ids)
        rec.update(saved(r))
        cases.append(rec)
    return {"cases": cases}


def dumps(data):
    """Compact JSON, one entry of every top-level list per line."""
    one = lambda v: json.dumps(v, ensure_ascii=False, separators=(",", ":"))  # noqa: E731
    items = [f"{one(k)}:" + ("[\n" + ",\n".join(map(one, v)) + "\n]" if isinstance(v, list) else one(v)) for k, v in data.items()]
    return "{\n" + ",\n".join(items) + "\n}"


def main(ref_root):
    sys.path.insert(0, os.path.abspath(ref_root))
    import minbpe as ref  # the reference
    assert os.path.abspath(os.path.dirname(ref.__file__)) == os.path.join(os.path.abspath(ref_root), "minbpe"), ref.__file__
    for name, data in (("golden_ref_suite.json", ref_suite(ref)), ("golden_fuzz_special.json", fuzz_special(ref)),
                       ("golden_fuzz_train.json", fuzz_train(ref))):
        with open(os.path.join(HERE, name), "w", encoding="utf-8") as f:
            f.write(dumps(data) + "\n")
    print("golden written to", HERE)


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(sys.argv[1])
