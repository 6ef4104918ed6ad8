"""
Host-side mirror of the minbpe API (reference: minbpe/base.py, basic.py, regex.py @1acefe8).

Same class names, method names, signatures, attributes and error behaviour as the reference,
so callers and the reference's own tests work unchanged; the loops underneath are not Python:

    train()            -> Engine.load_stream + Engine.train   (bpe_load_stream, bpe_train)
    encode*()          -> Engine.encode                        (bpe_encode)
    get_stats / merge  -> Engine.get_stats / Engine.merge      (bpe_get_stats, bpe_merge)
    GPT-4 pre-split    -> Engine.load_text_gpt4 / split_gpt4   (bpe_load_text_gpt4, bpe_split_gpt4) for texts
                          of at least 64 KiB; same chunks as regex.findall (tests/test_gpu_split.py)

What stays on the host, as in the reference: the regex pre-split for any other pattern and for
short texts (third-party ``regex`` module, regex.py:41,114), special-token splitting
(regex.py:123-164), vocab construction and the save/load file format (base.py:88-165), decode
(basic.py:51-55, regex.py:78-90).

There is no CPU fallback: without libb200bpe.so and a B200 the device-backed calls raise.
"""
import unicodedata

import numpy as np
import regex as re

from .engine import Engine

# tiktoken's split patterns, quoted by the reference at regex.py:18-19
GPT2_SPLIT_PATTERN = r"""'(?:[sdmt]|ll|ve|re)| ?\p{L}+| ?\p{N}+| ?[^\s\p{L}\p{N}]+|\s+(?!\S)|\s+"""
GPT4_SPLIT_PATTERN = r"""'(?i:[sdmt]|ll|ve|re)|[^\r\n\p{L}\p{N}]?+\p{L}+|\p{N}{1,3}| ?[^\s\p{L}\p{N}]++[\r\n]*|\s*[\r\n]|\s+(?!\S)|\s+"""

_shared_engine = None


def default_engine():
    """Process-wide engine used by the module-level get_stats/merge and by tokenizers that
    were not given a device."""
    global _shared_engine
    if _shared_engine is None:
        _shared_engine = Engine()
    return _shared_engine


# ---------------------------------------------------------------------------------------------
# base.py:13-41 — the two primitives, same signatures, computed on the GPU

def get_stats(ids, counts=None):
    """base.py:13-22.  Pair -> count over adjacent ids (overlaps counted); keys appear in
    first-occurrence order; an existing ``counts`` dict is updated in place and returned."""
    table = {} if counts is None else counts
    if len(ids) < 2:
        return table
    eng = default_engine()
    eng.load_ids(ids)
    pairs, cnt = eng.get_stats()
    for (p0, p1), c in zip(pairs.tolist(), cnt.tolist()):
        key = (p0, p1)
        table[key] = table.get(key, 0) + c
    return table


def merge(ids, pair, idx):
    """base.py:25-41.  New list with every left-to-right non-overlapping ``pair`` replaced."""
    if len(ids) == 0:
        return []
    eng = default_engine()
    eng.load_ids(ids)
    eng.merge(pair[0], pair[1], idx)
    return eng.read_stream().tolist()


# ---------------------------------------------------------------------------------------------
# base.py:44-61 — pretty printing helpers for the .vocab file

def replace_control_characters(s: str) -> str:
    """base.py:45-55: escape every code point whose Unicode category starts with 'C'."""
    return "".join(ch if unicodedata.category(ch)[0] != "C" else f"\\u{ord(ch):04x}" for ch in s)


def render_token(t: bytes) -> str:
    """base.py:57-61."""
    return replace_control_characters(t.decode("utf-8", errors="replace"))


def _batch_result(lists, flat):
    """encode_batch's two forms from per-document id lists: the lists, or (ids int32, offsets int64[len + 1])."""
    if not flat:
        return lists
    offsets = np.zeros(len(lists) + 1, dtype=np.int64)
    np.cumsum([len(x) for x in lists], out=offsets[1:])
    ids = np.fromiter((i for x in lists for i in x), dtype=np.int32, count=int(offsets[-1]))
    return ids, offsets


def _vocab_from_merges(merges, special_tokens):
    """base.py:88-95: 256 byte tokens, then merges in order, then specials."""
    vocab = {i: bytes((i,)) for i in range(256)}
    for (left, right), idx in merges.items():
        vocab[idx] = vocab[left] + vocab[right]
    for text, idx in special_tokens.items():
        vocab[idx] = text.encode("utf-8")
    return vocab


class Tokenizer:
    """base.py:66-165.  State: ``merges`` {(int,int): int}, ``pattern`` str, ``special_tokens``
    {str: int}, ``vocab`` {int: bytes}.  ``device`` (keyword only, not in the reference) picks the
    GPU; by default all tokenizers of a process share one engine on LOCAL_RANK / device 0."""

    def __init__(self, *, device=None):
        self.merges = {}
        self.pattern = ""
        self.special_tokens = {}
        self.vocab = self._build_vocab()
        self._device = device
        self._engine = None
        self._byte_perm = None     # 256-entry byte permutation applied before the merges (GPT4Tokenizer, gpt4.py:76-77)

    # -- device plumbing (not part of the reference API) --
    @property
    def engine(self):
        if self._engine is None:
            self._engine = default_engine() if self._device is None else Engine(self._device)
        return self._engine

    def _merge_array(self):
        # cached: built once per merges dict (a 32k-entry table costs ~10 ms of Python per encode call otherwise)
        n = len(self.merges)
        stamp = (id(self.merges), n, next(reversed(self.merges.items())) if n else None)
        if getattr(self, "_merge_cache", (None, None))[0] == stamp:
            return self._merge_cache[1]
        m = self._merge_array_build()
        self._merge_cache = (stamp, m)
        return m

    def _merge_array_build(self):
        m = np.empty((len(self.merges), 2), dtype=np.int32)
        for r, (pair, idx) in enumerate(self.merges.items()):
            if idx != 256 + r:
                raise ValueError("merges must map to consecutive ids starting at 256 in insertion order")
            m[r, 0], m[r, 1] = pair
        return m

    def _run_training(self, data, offsets, vocab_size, verbose, device_split=False, resume=False):
        """Shared by Basic/Regex: basic.py:21-49 / regex.py:37-70 minus the Python loops.  resume=True (not in the
        reference): keep the merges this tokenizer already has (e.g. from load()), replay them on the text and
        continue the same training run up to vocab_size — train(N) == train(k); save; load; train(N, resume=True)."""
        assert vocab_size >= 256
        num_merges = vocab_size - 256
        eng = self.engine
        if device_split:
            eng.load_text_gpt4(data)      # regex.py:41-44 on the GPU (k_split.cuh)
        else:
            eng.load_stream(data, offsets)
        have = None
        if resume and self.merges:
            have = self._merge_array()
            if len(have) > num_merges:
                raise ValueError(f"resume: the tokenizer already has {len(have)} merges, vocab_size {vocab_size} asks for fewer")
            eng.replay(have)
        k = 0 if have is None else len(have)
        pairs, counts, done = eng.train(num_merges - k, first_idx=256 + k)
        self.last_timing = eng.timing()
        if k:
            pairs = np.concatenate([have, pairs]) if done else have
            counts = np.concatenate([np.zeros(k, dtype=np.int64), counts]) if done else np.zeros(k, dtype=np.int64)
            done += k
        self._adopt(pairs, counts, done, num_merges, verbose, first_verbose=k)

    def _adopt(self, pairs, counts, done, num_merges, verbose, first_verbose=0):
        """basic.py:37-45: merges / vocab (and the verbose lines) from the pairs the device loop chose."""
        merges = {}
        vocab = {i: bytes((i,)) for i in range(256)}
        for i in range(done):
            pair = (int(pairs[i, 0]), int(pairs[i, 1]))
            idx = 256 + i
            merges[pair] = idx
            vocab[idx] = vocab[pair[0]] + vocab[pair[1]]
            if verbose and i >= first_verbose:
                print(f"merge {i+1}/{num_merges}: {pair} -> {idx} ({vocab[idx]}) had {int(counts[i])} occurrences")
        if done < num_merges:
            # the reference dies in max() on an empty stats dict (basic.py:35 / regex.py:56)
            # before it assigns self.merges / self.vocab
            raise ValueError("max() iterable argument is empty")
        self.merges = merges
        self.vocab = vocab

    # -- reference API --
    def train(self, text, vocab_size, verbose=False):
        raise NotImplementedError

    def encode(self, text):
        raise NotImplementedError

    def decode(self, ids):
        raise NotImplementedError

    def encode_batch(self, texts, *, flat=False):
        """[self.encode(t) for t in texts] (not in the reference).  flat=True: (ids int32, offsets int64 of len(texts) + 1)
        instead, document i being ids[offsets[i]:offsets[i + 1]]."""
        return _batch_result([self.encode(t) for t in texts], flat)

    def _build_vocab(self):
        return _vocab_from_merges(self.merges, self.special_tokens)

    # id lists at least this long are decoded on the GPU (bpe_decode) when this process already holds an engine
    # (decode is a host function in the reference and must keep working on a machine without a GPU, e.g. for a
    # model that was only loaded); same bytes as the joins below
    DEVICE_DECODE_MIN_IDS = 1 << 16

    def _decode_on_device(self, n_ids):
        return n_ids >= self.DEVICE_DECODE_MIN_IDS and (self._engine is not None or _shared_engine is not None)

    def _device_decode(self, ids, table):
        """table: {id: bytes}.  Returns (bytes, -1) or (None, position of the first id that is not in the table)."""
        top = max(table) + 1 if table else 0
        lens = np.full(top, 0xFFFFFFFF, dtype=np.uint32)
        starts = np.zeros(top, dtype=np.uint64)
        blob, pos = [], 0
        for idx, bts in table.items():
            if 0 <= idx < top:
                starts[idx], lens[idx] = pos, len(bts)
                blob.append(bts)
                pos += len(bts)
        arr = np.asarray(ids)
        if arr.dtype.kind not in "iu" or (arr.size and (arr.min() < -(2 ** 31) or arr.max() >= 2 ** 31)):
            return None, next(i for i, x in enumerate(ids) if not (isinstance(x, (int, np.integer)) and -(2 ** 31) <= x < 2 ** 31))
        return self.engine.decode(arr.astype(np.int32), np.frombuffer(b"".join(blob), dtype=np.uint8), starts, lens)

    def save(self, file_prefix):
        """base.py:97-138.  ``<prefix>.model`` (version, pattern, specials, one merge per line)
        and ``<prefix>.vocab`` (human readable, lossy)."""
        lines = ["minbpe v1", f"{self.pattern}", f"{len(self.special_tokens)}"]
        lines += [f"{text} {idx}" for text, idx in self.special_tokens.items()]
        lines += [f"{left} {right}" for left, right in self.merges]
        with open(file_prefix + ".model", "w") as f:  # default encoding, like base.py:106
            f.write("\n".join(lines) + "\n")
        parents = {idx: pair for pair, idx in self.merges.items()}
        with open(file_prefix + ".vocab", "w", encoding="utf-8") as f:
            for idx, token in self.vocab.items():
                shown = render_token(token)
                if idx in parents:
                    left, right = parents[idx]
                    f.write(f"[{render_token(self.vocab[left])}][{render_token(self.vocab[right])}] -> [{shown}] {idx}\n")
                else:
                    f.write(f"[{shown}] {idx}\n")

    def load(self, model_file):
        """base.py:140-165.  Merge ids are assigned 256, 257, ... by line order."""
        assert model_file.endswith(".model")
        merges, specials = {}, {}
        with open(model_file, "r", encoding="utf-8") as f:
            assert f.readline().strip() == "minbpe v1"
            self.pattern = f.readline().strip()
            for _ in range(int(f.readline().strip())):
                text, idx = f.readline().strip().split()
                specials[text] = int(idx)
            for idx, line in enumerate(f, start=256):
                left, right = map(int, line.split())
                merges[(left, right)] = idx
        self.merges = merges
        self.special_tokens = specials
        self.vocab = self._build_vocab()


class BasicTokenizer(Tokenizer):
    """basic.py:15-74: the whole text is one id stream (one chunk)."""

    def __init__(self, *, device=None):
        super().__init__(device=device)

    def train(self, text, vocab_size, verbose=False, *, resume=False):
        assert vocab_size >= 256
        self._run_training(text.encode("utf-8"), None, vocab_size, verbose, resume=resume)

    def decode(self, ids):
        if self._decode_on_device(len(ids)):
            data, bad = self._device_decode(ids, self.vocab)
            if data is None:
                raise KeyError(ids[bad])          # what self.vocab[idx] raises (basic.py:53)
            return data.decode("utf-8", errors="replace")
        return b"".join(self.vocab[idx] for idx in ids).decode("utf-8", errors="replace")

    def encode(self, text):
        data = text.encode("utf-8")
        if len(data) < 2 or not self.merges:
            return list(data)
        return self.engine.encode(data, None, self._merge_array(), self._byte_perm).tolist()


def split_text(compiled_pattern, text):
    """regex.py:41-44 as arrays: (utf-8 bytes of all chunks back to back, start offset of every
    chunk).  When the matches tile the text (always true for the GPT-2/GPT-4 patterns) the
    bytes are just text.encode() and offsets come from the match lengths."""
    chunks = compiled_pattern.findall(text)
    if not chunks:
        return b"", np.zeros(0, dtype=np.uint64)
    char_len = np.fromiter(map(len, chunks), dtype=np.int64, count=len(chunks))
    if int(char_len.sum()) == len(text) and int(char_len.min()) > 0:
        data = text.encode("utf-8")
        char_off = np.zeros(len(chunks), dtype=np.int64)
        np.cumsum(char_len[:-1], out=char_off[1:])
        if len(data) == len(text):
            return data, char_off.astype(np.uint64)
        raw = np.frombuffer(data, dtype=np.uint8)
        char_start = np.flatnonzero((raw & 0xC0) != 0x80)  # byte index of every code point
        return data, char_start[char_off].astype(np.uint64)
    # general pattern: matches may skip text or be empty
    enc = [c.encode("utf-8") for c in chunks]
    enc = [c for c in enc if c]
    lens = np.fromiter(map(len, enc), dtype=np.int64, count=len(enc))
    offs = np.zeros(len(enc), dtype=np.int64)
    if len(enc) > 1:
        np.cumsum(lens[:-1], out=offs[1:])
    return b"".join(enc), offs.astype(np.uint64)


class RegexTokenizer(Tokenizer):
    """regex.py:22-164: regex pre-split into chunks; pairs and merges never cross a chunk."""

    def __init__(self, pattern=None, *, device=None):
        super().__init__(device=device)
        self.pattern = GPT4_SPLIT_PATTERN if pattern is None else pattern
        self.compiled_pattern = re.compile(self.pattern)
        self.special_tokens = {}
        self.inverse_special_tokens = {}

    # texts at least this long are split on the GPU when the pattern is the GPT-4 one (same chunks as
    # regex.findall — tests/test_split_rules.py, tests/test_gpu_split.py); short ones stay on the host
    DEVICE_SPLIT_MIN_BYTES = 1 << 16

    _DEVICE_PATTERNS = {GPT4_SPLIT_PATTERN: 0, GPT2_SPLIT_PATTERN: 1}     # BPE_OPT_SPLIT_PATTERN values

    def _device_split(self, nbytes):
        """Large texts under one of the reference's two patterns (regex.py:18-19) are split on the GPU; the engine may be
        shared by tokenizers with different patterns, so the pattern is selected before every such call."""
        # the pattern that is actually used for splitting is compiled_pattern (regex.py:32,41,114), not the
        # `pattern` string, which load() may have replaced
        which = self._DEVICE_PATTERNS.get(self.compiled_pattern.pattern)
        if which is None or nbytes < self.DEVICE_SPLIT_MIN_BYTES:
            return False
        from .engine import OPT_SPLIT_PATTERN
        self.engine.set_option(OPT_SPLIT_PATTERN, which)
        return True

    def _device_specials(self, special):
        """The device front end takes at most 64 specials of 1..48 utf-8 bytes and non-negative int32 ids; anything else
        keeps the reference's host split (below)."""
        E = Engine
        return (0 < len(special) <= E.SPECIAL_MAX and
                all(isinstance(k, str) and 0 < len(k.encode("utf-8")) <= E.SPECIAL_MAX_BYTES and 0 <= int(v) < 2 ** 31 for k, v in special.items()))

    def train(self, text, vocab_size, verbose=False, *, resume=False):
        assert vocab_size >= 256
        data = text.encode("utf-8")
        if self._device_split(len(data)):
            self._run_training(data, None, vocab_size, verbose, device_split=True, resume=resume)
            return
        data, offsets = split_text(self.compiled_pattern, text)
        self._run_training(data, offsets, vocab_size, verbose, resume=resume)

    def train_from_file(self, path, vocab_size, verbose=False, *, group=None):
        """train() for a UTF-8 text file of any size (not in the reference, which takes a str: regex.py:36).  The file
        is memory-mapped and split on the device in pieces; when torch.distributed is initialised (one process per
        GPU) every rank trains on its own byte range — cut where a letter is followed by a space, a provable chunk
        boundary of both patterns — and all ranks end with identical merges / vocab.  GPT-2 / GPT-4 split patterns only."""
        assert vocab_size >= 256
        which = self._DEVICE_PATTERNS.get(self.compiled_pattern.pattern)
        if which is None:
            raise ValueError("train_from_file splits on the device and supports the GPT-2 / GPT-4 split patterns only; "
                             "use train(open(path).read(), ...) for other patterns")
        from .dist import train_file
        from .engine import OPT_SPLIT_PATTERN
        eng = self.engine
        eng.set_option(OPT_SPLIT_PATTERN, which)
        pairs, counts, done = train_file(eng, eng.device, path, vocab_size - 256, group=group)
        self.last_timing = eng.timing()
        self._adopt(pairs, counts, done, vocab_size - 256, verbose)

    def encode_file(self, path, allowed_special="none", *, group=None, gather=False):
        """encode() for a UTF-8 text file of any size (not in the reference, which takes a str: regex.py:123): the file is
        memory-mapped; with torch.distributed initialised every rank encodes its own byte range and returns its own ids
        (rank order = text order; gather=True concatenates them on rank 0).  GPT-2 / GPT-4 split patterns, special tokens
        within the limits of the device front end.  "none_raise" is not offered: it would scan the file on the host."""
        which = self._DEVICE_PATTERNS.get(self.compiled_pattern.pattern)
        if which is None:
            raise ValueError("encode_file splits on the device and supports the GPT-2 / GPT-4 split patterns only")
        if allowed_special == "all":
            special = self.special_tokens
        elif allowed_special == "none":
            special = {}
        elif isinstance(allowed_special, set):
            special = {k: v for k, v in self.special_tokens.items() if k in allowed_special}
        else:
            raise ValueError(f"allowed_special={allowed_special} not understood (encode_file takes 'all', 'none' or a set)")
        if special and not self._device_specials(special):
            raise ValueError("encode_file needs special tokens the device front end takes (at most 64, 1..48 utf-8 bytes each)")
        from .dist import encode_file
        from .engine import OPT_SPLIT_PATTERN
        eng = self.engine
        eng.set_option(OPT_SPLIT_PATTERN, which)
        spec = [(k.encode("utf-8"), int(v)) for k, v in special.items()] or None
        return encode_file(eng, path, self._merge_array(), self._byte_perm, spec, group=group, gather=gather)

    def register_special_tokens(self, special_tokens):
        self.special_tokens = special_tokens
        self.inverse_special_tokens = {idx: text for text, idx in special_tokens.items()}

    def decode(self, ids):
        if self._decode_on_device(len(ids)):
            table = {idx: text.encode("utf-8") for idx, text in self.inverse_special_tokens.items()}
            table.update(self.vocab)              # regex.py:81-86: the vocabulary first, then the special tokens
            data, bad = self._device_decode(ids, table)
            if data is None:
                raise ValueError(f"invalid token id: {ids[bad]}")
            return data.decode("utf-8", errors="replace")
        parts = []
        for idx in ids:
            if idx in self.vocab:
                parts.append(self.vocab[idx])
            elif idx in self.inverse_special_tokens:
                parts.append(self.inverse_special_tokens[idx].encode("utf-8"))
            else:
                raise ValueError(f"invalid token id: {idx}")
        return b"".join(parts).decode("utf-8", errors="replace")

    def _encode_chunk(self, text_bytes):
        """regex.py:92-109 for a single chunk."""
        if not self.merges or (len(text_bytes) < 2 and self._byte_perm is None):
            return list(text_bytes)
        return self.engine.encode(bytes(text_bytes), None, self._merge_array(), self._byte_perm).tolist()

    def encode_ordinary(self, text):
        """regex.py:111-121."""
        raw = text.encode("utf-8")
        if self.merges and self._device_split(len(raw)):
            return self.engine.encode_text_gpt4(raw, self._merge_array(), self._byte_perm).tolist()   # split + encode on the device, no offsets
        data, offsets = split_text(self.compiled_pattern, text)
        if not self.merges or (len(data) < 2 and self._byte_perm is None):
            return list(data)
        if not len(data):
            return []
        return self.engine.encode(data, offsets, self._merge_array(), self._byte_perm).tolist()

    def encode_ordinary_batch(self, texts, *, flat=False):
        """[self.encode_ordinary(t) for t in texts] (not in the reference); flat as in encode_batch.  Batches of at least
        DEVICE_SPLIT_MIN_BYTES under the GPT-2 / GPT-4 pattern are split and encoded in one device call."""
        return self._encode_batch(texts, None, flat)

    def encode_batch(self, texts, allowed_special="none_raise", *, flat=False):
        """[self.encode(t, allowed_special) for t in texts] (not in the reference): same ids, same errors.  flat=True:
        (ids int32, offsets int64 of len(texts) + 1), document i being ids[offsets[i]:offsets[i + 1]] — no Python list per
        id.  Batches of at least DEVICE_SPLIT_MIN_BYTES under the GPT-2 / GPT-4 pattern, with special tokens the device
        front end takes, are split and encoded in one device call (bpe_encode_batch_gpt4); others loop over encode()."""
        return self._encode_batch(texts, allowed_special, flat)

    def _encode_batch(self, texts, allowed_special, flat):
        texts = list(texts)
        if not texts:
            return _batch_result([], flat)
        if allowed_special is None:
            special, one = {}, self.encode_ordinary
        else:
            special = self._resolve_special(allowed_special)
            one = lambda t: self.encode(t, allowed_special)     # noqa: E731
        if not self.merges or (special and not self._device_specials(special)):
            return _batch_result([one(t) for t in texts], flat)
        raws = []
        for t in texts:      # encode()'s checks, document by document: the first failing document raises what the loop would
            if allowed_special == "none_raise":
                assert all(token not in t for token in self.special_tokens)
            raws.append(t.encode("utf-8"))
        if not self._device_split(sum(map(len, raws))):
            return _batch_result([one(t) for t in texts], flat)
        spec = [(k.encode("utf-8"), int(v)) for k, v in special.items()] or None
        ids, offsets = self.engine.encode_batch_gpt4(b"\xff".join(raws), len(raws), self._merge_array(), self._byte_perm, specials=spec)
        if flat:
            return ids, offsets
        flat_ids, o = ids.tolist(), offsets.tolist()
        return [flat_ids[o[i]:o[i + 1]] for i in range(len(raws))]

    def _resolve_special(self, allowed_special):
        """regex.py:131-145: the specials allowed_special selects ("none_raise": none; the caller checks the text)."""
        if allowed_special == "all":
            return self.special_tokens
        if allowed_special in ("none", "none_raise"):
            return {}
        if isinstance(allowed_special, set):
            return {k: v for k, v in self.special_tokens.items() if k in allowed_special}
        raise ValueError(f"allowed_special={allowed_special} not understood")

    def encode(self, text, allowed_special="none_raise"):
        """regex.py:123-164."""
        special = self._resolve_special(allowed_special)
        if allowed_special == "none_raise":
            assert all(token not in text for token in self.special_tokens)
        if not special:
            return self.encode_ordinary(text)
        if self.merges and self._device_specials(special):
            raw = text.encode("utf-8")
            if self._device_split(len(raw)):
                # regex.py:152-163 on the GPU: the specials are found there, every part between them is split and encoded
                # on its own, one call (k_special.cuh)
                spec = [(k.encode("utf-8"), int(v)) for k, v in special.items()]
                return self.engine.encode_text_gpt4(raw, self._merge_array(), self._byte_perm, specials=spec).tolist()
        splitter = "(" + "|".join(re.escape(k) for k in special) + ")"
        ids = []
        for part in re.split(splitter, text):
            if part in special:
                ids.append(special[part])
            else:
                ids.extend(self.encode_ordinary(part))
        return ids
