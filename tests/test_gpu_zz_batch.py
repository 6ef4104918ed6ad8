"""GPU: batched encode (bpe_encode_batch_gpt4, RegexTokenizer.encode_batch / encode_ordinary_batch): many documents in one
device call give exactly the ids of encoding every document on its own — against the reference's per-document procedure
(re.split at the specials + split + _encode_chunk) restated with the oracle, against the per-document loop of the classes,
and against the unmodified reference class's recorded answers."""
import hashlib
import os
import random

import numpy as np
import pytest
import regex

import oracle
from conftest import load_golden
from minbpe_b200 import engine as E
from minbpe_b200.tokenizer import GPT2_SPLIT_PATTERN, GPT4_SPLIT_PATTERN

pytestmark = pytest.mark.gpu

SMALL = bool(os.environ.get("BPE_TEST_SMALL"))      # set when the suite runs on the CPU SIMT emulator
PATTERNS = {0: regex.compile(GPT4_SPLIT_PATTERN), 1: regex.compile(GPT2_SPLIT_PATTERN)}
ALPHABET = list("ab'sSdDmMtTlLvVeErR 12\t\n\r!.,' 　é日ſ½") + ["  ", "\n\n", "'ll", "'ve", " '", "the ", "ing", "\U0001f600"]
SPECIAL_SETS = [["<|endoftext|>"], ["<|a|>", "<|ab|>", "|>"], [" <s> ", "'s", "12"], ["x", "日"], ["\n<eot>\n", "  "], ["a b", "b a"]]
# pairs whose concatenation splits differently from the two texts: trailing spaces, a contraction, digit groups, CR LF,
# a space before punctuation
SEAMS = [("a  ", "  b"), ("don'", "t"), ("12", "345"), ("\r", "\n"), ("x ", "!"), ("a\n", "\nb"), ("'", "ll"), (" ", " ")]


def ref_encode(text, special, merges, pattern=0, perm=None):
    """regex.py:152-163 for one document, with oracle.c_encode as encode_ordinary"""
    parts = regex.split("(" + "|".join(regex.escape(k) for k in special) + ")", text) if special else [text]
    out = []
    for part in parts:
        if special and part in special:
            out.append(special[part])
        elif part:
            d, o = oracle.split_to_stream(part, PATTERNS[pattern])
            out.extend(oracle.c_encode(d, o, merges, perm).tolist())
    return out


def split_docs(ids, offsets):
    ids = ids.tolist()
    return [ids[offsets[i]:offsets[i + 1]] for i in range(len(offsets) - 1)]


def sha(ids):
    return hashlib.sha256(np.asarray(ids, dtype="<i4").tobytes()).hexdigest()


@pytest.fixture(scope="module")
def tok():
    from minbpe_b200 import RegexTokenizer
    from minbpe_b200.synth import generate
    text = generate(1337, 1 << 20).tobytes().decode("utf-8")[:300000]
    t = RegexTokenizer()
    t.train(text, 256 + 200)
    t.text = text
    t.m = np.array(list(t.merges.keys()), dtype=np.int32)
    return t


def random_doc(rnd, names):
    parts = []
    for _ in range(rnd.randint(0, 6)):
        parts.append("".join(rnd.choice(ALPHABET) for _ in range(rnd.randint(0, 12))))
        if names and rnd.random() < 0.5:
            parts.append(rnd.choice(names))
    return "".join(parts)


def test_random_batches_through_the_abi(tok):
    """(a) 300 seeded batches of 1..40 adversarial documents, both patterns, with and without specials"""
    eng = E.Engine(0)
    rnd = random.Random(1234)
    n_docs_seen = 0
    for it in range(300):
        pattern = it % 2
        names = rnd.choice(SPECIAL_SETS) if it % 3 else []
        special = {k: 100000 + i for i, k in enumerate(names)}
        docs = []
        for _ in range(rnd.randint(1, 40)):
            r = rnd.random()
            if r < 0.15:
                docs.append("")
            elif r < 0.3:
                docs.append(rnd.choice(rnd.choice(SEAMS)))
            elif r < 0.4 and names:
                docs.append(rnd.choice(names))                          # a document that is one special token
            else:
                docs.append(random_doc(rnd, names))
        if it % 5 == 0:
            docs = [""] + docs + [""]                                     # empty documents at both ends
        if it % 7 == 0:
            a, b = SEAMS[(it // 7) % len(SEAMS)]
            docs = docs + [a, b] + [a, "", b]
        eng.set_option(E.OPT_SPLIT_PATTERN, pattern)
        spec = [(k.encode("utf-8"), v) for k, v in special.items()] or None
        data = b"\xff".join(d.encode("utf-8") for d in docs)
        ids, offs = eng.encode_batch_gpt4(data, len(docs), tok.m, specials=spec)
        assert offs[0] == 0 and offs[-1] == len(ids) and np.all(np.diff(offs) >= 0)
        got = split_docs(ids, offs)
        for d, doc in enumerate(docs):
            assert got[d] == ref_encode(doc, special, tok.m, pattern), (it, d, doc, names, pattern)
        n_docs_seen += len(docs)
    eng.set_option(E.OPT_SPLIT_PATTERN, 0)
    assert n_docs_seen > 3000
    eng.close()


def _docs_with_specials(tok, rnd, n, names):
    out = []
    for i in range(n):
        lo = rnd.randrange(0, len(tok.text) - 3000)
        body = tok.text[lo:lo + rnd.randint(0, 2500)]
        if names and i % 3 == 0:
            cut = rnd.randint(0, len(body))
            body = body[:cut] + rnd.choice(names) + body[cut:]
        out.append(body)
    return out


def _synthetic_gpt4_tokenizer():
    from minbpe_b200 import GPT4Tokenizer
    from test_gpt4_host import synthetic_ranks
    with open(os.path.join(os.path.dirname(__file__), "golden", "taylorswift.txt"), encoding="utf-8") as f:
        ts = f.read()
    ranks, merges, perm = synthetic_ranks(ts[:30000], 120)
    return GPT4Tokenizer(mergeable_ranks=ranks)


def test_classes_equal_the_per_document_loop(tok):
    """(b) encode_batch / encode_ordinary_batch == the loop over encode / encode_ordinary, every allowed_special mode"""
    from minbpe_b200 import RegexTokenizer
    rnd = random.Random(5)
    sp = {"<|endoftext|>": 100257, "<|fim_prefix|>": 100258, " <sp> ": 100259}
    toks = []
    for pattern in (GPT4_SPLIT_PATTERN, GPT2_SPLIT_PATTERN, r"\w+|\s+|[^\w\s]+"):   # the last one: no device split, the loop
        t = RegexTokenizer(pattern)
        t.merges = dict(tok.merges)
        t.vocab = t._build_vocab()
        toks.append(t)
    toks.append(_synthetic_gpt4_tokenizer())
    for t in toks:
        t.DEVICE_SPLIT_MIN_BYTES = 0
        t.register_special_tokens({**t.special_tokens, **sp})
        names = list(sp)
        docs = [""] + _docs_with_specials(tok, rnd, 25, names) + ["", "<|endoftext|>", "don'", "t", ""]
        plain = [d for d in docs if not any(k in d for k in t.special_tokens)]
        for mode in ("all", "none", {"<|fim_prefix|>"}, set()):
            want = [t.encode(d, allowed_special=mode) for d in docs]
            assert t.encode_batch(docs, allowed_special=mode) == want, (t.pattern[:10], mode)
            ids, offs = t.encode_batch(docs, allowed_special=mode, flat=True)
            assert ids.dtype == np.int32 and offs.dtype == np.int64 and len(offs) == len(docs) + 1
            assert split_docs(ids, offs) == want
        assert t.encode_batch(plain) == [t.encode(d) for d in plain]
        assert t.encode_ordinary_batch(docs) == [t.encode_ordinary(d) for d in docs]
        with pytest.raises(AssertionError):
            t.encode_batch(docs)                                           # "none_raise" with a special in the batch
        with pytest.raises(ValueError):
            t.encode_batch(docs, allowed_special="bogus")
        with pytest.raises(UnicodeEncodeError):
            t.encode_batch(["abc", "x\ud800y"], allowed_special="all")
        with pytest.raises(AttributeError):
            t.encode_ordinary_batch(["abc", 7])
        assert t.encode_batch([]) == [] and t.encode_ordinary_batch([]) == []
        ids, offs = t.encode_batch([], flat=True)
        assert ids.size == 0 and offs.tolist() == [0]
        # specials the device front end does not take (longer than 48 bytes) keep the loop: same answer
        long_sp = {**t.special_tokens, "<|" + "y" * 60 + "|>": 100300}
        t.register_special_tokens(long_sp)
        docs2 = docs + ["a<|" + "y" * 60 + "|>b"]
        assert t.encode_batch(docs2, allowed_special="all") == [t.encode(d, allowed_special="all") for d in docs2]
    # the reference's default threshold: a small batch goes through the loop, a large one through the device
    t = toks[0]
    t.DEVICE_SPLIT_MIN_BYTES = RegexTokenizer.DEVICE_SPLIT_MIN_BYTES
    for docs in (["hello world", "", "don't"], _docs_with_specials(tok, rnd, 80, [])):
        assert t.encode_ordinary_batch(docs) == [t.encode_ordinary(d) for d in docs]
    # the same batch against the oracle
    docs = _docs_with_specials(tok, rnd, 30, list(sp))
    t.DEVICE_SPLIT_MIN_BYTES = 0
    t.register_special_tokens(sp)
    assert t.encode_batch(docs, allowed_special="all") == [ref_encode(d, sp, tok.m) for d in docs]


def test_documents_straddle_pieces_and_fall_back(tok):
    """(c) small pieces: documents straddle many piece cuts; a 12,000-letter chunk makes exactly one fall-back piece"""
    eng = E.Engine(0)
    rnd = random.Random(77)
    sp = {"<|im start|>": 9001, "d e": 9002}
    spec = [(k.encode("utf-8"), v) for k, v in sp.items()]
    docs = _docs_with_specials(tok, rnd, 60, list(sp))
    docs[10] = tok.text[:40000]                                          # longer than several pieces: letter+space cuts
    docs[11] = ""
    want = [ref_encode(d, sp, tok.m) for d in docs]
    data = b"\xff".join(d.encode("utf-8") for d in docs)
    eng.set_option(E.OPT_SPLIT_PIECE, 1 << 14)
    try:
        ids, offs = eng.encode_batch_gpt4(data, len(docs), tok.m, specials=spec)
        assert split_docs(ids, offs) == want
        assert eng.encode_stats()["pieces"] > 5
    finally:
        eng.set_option(E.OPT_SPLIT_PIECE, 0)
    docs2 = docs[:20] + [tok.text[:3000] + " " + "lyiltumdya" * 1200 + " d e" + tok.text[3000:6000], "", "<|im start|>"] + docs[20:40]
    data2 = b"\xff".join(d.encode("utf-8") for d in docs2)
    ids, offs = eng.encode_batch_gpt4(data2, len(docs2), tok.m, specials=spec)
    assert split_docs(ids, offs) == [ref_encode(d, sp, tok.m) for d in docs2]
    assert eng.encode_stats()["fallback_pieces"] == 1
    ids, offs = eng.encode_batch_gpt4(data, len(docs), tok.m, specials=spec)    # and the memo works again
    assert split_docs(ids, offs) == want
    assert eng.encode_stats()["fallback_pieces"] == 0
    eng.close()


def test_golden_fuzz_cases_as_batches():
    """(d) every recorded answer of the reference class, as the batch [text, "", text]"""
    from minbpe_b200 import RegexTokenizer
    g = load_golden("golden_fuzz_special.json")
    toks = {}
    for name, pat in (("gpt4", GPT4_SPLIT_PATTERN), ("gpt2", GPT2_SPLIT_PATTERN)):
        o = RegexTokenizer(pat)
        o.merges = {(a, b): 256 + i for i, (a, b) in enumerate(g["merges"][name])}
        o.vocab = o._build_vocab()
        o.DEVICE_SPLIT_MIN_BYTES = 0
        toks[name] = o
    n = 0
    for it, c in enumerate(g["cases"]):
        o, text = toks[c["pattern"]], c["text"]
        o.register_special_tokens(c["special"])
        allowed = c["allowed"] if c["allowed"] == "all" else set(c["allowed"])
        o.engine.set_option(E.OPT_SPLIT_PIECE, c["piece"])
        try:
            try:
                got = o.encode_batch([text, "", text], allowed_special=allowed)
            except E.EngineError as ex:          # a tiny piece size may find no cut point: a clean error, not a wrong answer
                assert "cut point" in str(ex), ex
                continue
        finally:
            o.engine.set_option(E.OPT_SPLIT_PIECE, 0)
        want = (c["n_ids"], c["ids_sha256"])
        assert [(len(x), sha(x)) for x in got] == [want, (0, sha([])), want], (it, c["pattern"], text)
        n += 1
    assert n >= len(g["cases"]) // 2


def test_encode_and_encode_batch_share_the_memo(tok):
    """(e) same merges: encode, encode_batch, encode — the repeat adds no chunk to the memo"""
    from minbpe_b200 import RegexTokenizer
    t = RegexTokenizer()
    t.merges = dict(tok.merges)
    t.vocab = t._build_vocab()
    text = tok.text[:120000]
    docs = [text[i:i + 3000] for i in range(0, len(text), 3000)]
    first = t.encode(text)
    assert t.engine.encode_stats()["new_chunks"] > 0
    batch = t.encode_batch(docs)
    assert batch == [ref_encode(d, {}, tok.m) for d in docs]
    assert t.engine.encode_stats()["fallback_pieces"] == 0
    assert t.encode(text) == first
    assert t.engine.encode_stats()["new_chunks"] == 0          # the batch neither reset nor replaced the memo


def test_separator_count_and_capacity_errors(tok):
    """(f) bytes that do not hold n_docs - 1 separators, and an output buffer that is too small, are errors"""
    import ctypes
    eng = E.Engine(0)
    eng.set_option(E.OPT_SPLIT_PATTERN, 0)
    with pytest.raises(E.EngineError, match="separators"):
        eng.encode_batch_gpt4(b"abc\xffdef", 3, tok.m)
    with pytest.raises(E.EngineError, match="separators"):
        eng.encode_batch_gpt4(b"abc\xffdef\xff\xffx", 3, tok.m)
    with pytest.raises(E.EngineError):
        eng.encode_batch_gpt4(b"abc", 0, tok.m)
    ids, offs = eng.encode_batch_gpt4(b"", 1, tok.m)
    assert ids.size == 0 and offs.tolist() == [0, 0]
    ids, offs = eng.encode_batch_gpt4(b"\xff\xff", 3, tok.m)
    assert ids.size == 0 and offs.tolist() == [0, 0, 0, 0]
    data = np.frombuffer(b"hello world\xffhow are you", dtype=np.uint8)
    m = np.ascontiguousarray(tok.m)
    out = np.empty(3, dtype=np.int32)
    doc = np.zeros(3, dtype=np.uint64)
    n = ctypes.c_uint64()
    rc = eng._lib.bpe_encode_batch_gpt4(eng._h, E._ptr(data), data.size, 2, E._ptr(m), m.shape[0], None, None, None, None, 0,
                                        E._ptr(out), out.size, ctypes.byref(n), E._ptr(doc))
    assert rc == E.ERR_CAPACITY
    with pytest.raises(E.EngineError, match="too small"):
        eng._check(rc, "bpe_encode_batch_gpt4")
    eng.close()


@pytest.mark.skipif(SMALL, reason="256 MiB: too large for the CPU SIMT emulator")
def test_large_batch(tok):
    """(g) 256 MiB of synthetic text as ~10^5 documents: offsets monotone, ending at out_n; a seeded sample equals the oracle"""
    from minbpe_b200.synth import generate
    raw = generate(2024, 256 << 20).tobytes()
    text = raw.decode("utf-8")
    rnd = random.Random(3)
    cuts = sorted(rnd.sample(range(1, len(text)), 100000 - 1))
    docs = [text[a:b] for a, b in zip([0] + cuts, cuts + [len(text)])]
    eng = E.Engine(0)
    eng.set_option(E.OPT_SPLIT_PATTERN, 0)
    data = b"\xff".join(d.encode("utf-8") for d in docs)
    ids, offs = eng.encode_batch_gpt4(data, len(docs), tok.m)
    assert len(offs) == len(docs) + 1 and offs[0] == 0 and offs[-1] == len(ids) and np.all(np.diff(offs) >= 0)
    for d in sorted(rnd.sample(range(len(docs)), 500)):
        assert ids[offs[d]:offs[d + 1]].tolist() == ref_encode(docs[d], {}, tok.m), d
    eng.close()
