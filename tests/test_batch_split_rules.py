"""CPU: the split rules of the batched encode (k_batch.cuh).  Documents joined by single 0xFF bytes, every separator a
one-byte boundary occurrence (class SC_B, as a special token's bytes get), give exactly the per-document splits of
`regex` — for both patterns, at several tile sizes, with empty documents, across every seam where joining the texts
themselves would change the split, and with special tokens inside the documents (hits = separators + specials)."""
import random

import numpy as np
import regex

import oracle
from minbpe_b200.tokenizer import GPT2_SPLIT_PATTERN, GPT4_SPLIT_PATTERN
from minbpe_b200.unicode_tables import tables

GPT4, GPT2 = regex.compile(GPT4_SPLIT_PATTERN), regex.compile(GPT2_SPLIT_PATTERN)
ALPHABET = list("ab'sSdDmMtTlLvVeErR 12\t\n\r!.,' 　é日ſ½") + ["  ", "\n\n", "'ll", "'ve", " '", "K", "\U0001f600"]
SPECIAL_SETS = [["<|endoftext|>"], ["<|a|>", "<|ab|>", "|>"], [" <s> ", "'s", "12"], ["x", "日"], ["\n<eot>\n", "  "], ["a b", "b a"]]
# seams where split(a + b) != split(a) + split(b): trailing spaces, a contraction, digit groups, CR LF, space + punctuation
SEAMS = [("a  ", "  b"), ("don'", "t"), ("12", "345"), ("1", "2"), ("\r", "\n"), ("x ", "!"), ("  ", ""), ("", "'s"),
         ("a\n", "\nb"), ("9 ", "9"), ("é", "日"), ("'", "ll"), ("\t", " \t"), (" ", " ")]


def expected(docs, pattern, specials=()):
    """per-document re.split at the specials + findall, plus a one-byte occurrence per separator"""
    offs, hits, pos = [], [], 0
    pat = regex.compile("(" + "|".join(regex.escape(k) for k in specials) + ")") if specials else None
    for d, doc in enumerate(docs):
        if d:
            offs.append(pos)
            hits.append((pos, 1))
            pos += 1
        for part in (pat.split(doc) if pat else [doc]):
            nb = len(part.encode("utf-8"))
            if specials and part in specials:
                offs.append(pos)
                hits.append((pos, nb))
            else:
                p = pos
                for ch in pattern.findall(part):
                    offs.append(p)
                    p += len(ch.encode("utf-8"))
            pos += nb
    return np.asarray(offs, dtype=np.uint64), hits


def check(docs, tiles, specials=()):
    cls, contr = tables()
    data = b"\xff".join(d.encode("utf-8") for d in docs)
    if not data:
        return 0
    n = 0
    for pattern, fn in ((GPT4, oracle.split_logic_offsets_special), (GPT2, oracle.split_logic_offsets_gpt2)):
        want, hits = expected(docs, pattern, specials)
        for tile in tiles:
            got = fn(data, cls, contr, hits, tile)
            assert np.array_equal(got, want), (docs, specials, pattern.pattern[:12], tile, got.tolist(), want.tolist())
            n += 1
    return n


def test_seams():
    for a, b in SEAMS:
        assert GPT4.findall(a + b) != GPT4.findall(a) + GPT4.findall(b) or GPT2.findall(a + b) != GPT2.findall(a) + GPT2.findall(b) \
            or not (a and b), (a, b)
        check([a, b], (0, 1, 2, 3, 5))
        check(["", a, "", b, ""], (0, 1, 4))
        check([b, a, b], (0, 2, 7))


def test_random_batches_with_empty_documents():
    rnd = random.Random(4242)
    n = 0
    for _ in range(3000):
        docs = []
        for _ in range(rnd.randint(1, 6)):
            r = rnd.random()
            if r < 0.2:
                docs.append("")
            elif r < 0.4:
                docs.append(rnd.choice(rnd.choice(SEAMS)))
            else:
                docs.append("".join(rnd.choice(ALPHABET) for _ in range(rnd.randint(1, 12))))
        n += check(docs, (0, rnd.randint(1, 9)))
    assert n > 10000


def test_random_batches_with_specials_inside_documents():
    rnd = random.Random(777)
    n = 0
    for _ in range(2000):
        specials = rnd.choice(SPECIAL_SETS)
        docs = []
        for _ in range(rnd.randint(1, 5)):
            parts = []
            for _ in range(rnd.randint(0, 4)):
                parts.append("".join(rnd.choice(ALPHABET) for _ in range(rnd.randint(0, 10))))
                if rnd.random() < 0.6:
                    parts.append(rnd.choice(specials))
            docs.append("".join(parts))
        n += check(docs, (0, rnd.randint(1, 9)), specials)
    assert n > 6000
