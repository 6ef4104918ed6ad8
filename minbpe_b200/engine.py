"""
ctypes binding of libb200bpe.so (include/b200bpe.h) — the only door between the Python host
classes and the sm_100a kernels.  There is NO CPU fallback: if the library is missing or no
B200 is present, every operation raises.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BPE_LIB_PATH") or os.path.join(_HERE, "csrc", "libb200bpe.so")  # override: A/B builds
ABI_VERSION = 1

OPT_KERNEL_TIMING, OPT_RESCAN, OPT_BATCH, OPT_TABLE_LOG2, OPT_SPLIT_PIECE, OPT_VOCAB_CAP, OPT_ENC_MEMO_LOG2, OPT_SPLIT_PATTERN, OPT_HIST_KERNEL, OPT_SEG_FILTER = 1, 2, 3, 4, 5, 6, 7, 8, 9, 10
ERR_CAPACITY = -4

_lib = None


class EngineError(RuntimeError):
    pass


class Timing(ctypes.Structure):
    _fields_ = [("loop_ms", ctypes.c_double), ("init_ms", ctypes.c_double), ("merge_kernel_ms", ctypes.c_double),
                ("tokens_in", ctypes.c_uint64), ("tokens_out", ctypes.c_uint64), ("kernel_launches", ctypes.c_uint64),
                ("table_slots", ctypes.c_uint64), ("table_used", ctypes.c_uint64), ("h2d_bytes", ctypes.c_uint64),
                ("d2h_bytes", ctypes.c_uint64), ("hist_kernel", ctypes.c_uint64),
                ("filter_candidates", ctypes.c_uint64), ("filter_segments", ctypes.c_uint64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


def load_library():
    """Load libb200bpe.so and declare every entry point of include/b200bpe.h."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise EngineError(f"{LIB_PATH} not found: build it with `python minbpe_b200/csrc/build.py` "
                          "(minbpe_b200 has no CPU fallback)")
    L = ctypes.CDLL(LIB_PATH)
    vp, u64, i32, i64, ci = ctypes.c_void_p, ctypes.c_uint64, ctypes.c_int32, ctypes.c_int64, ctypes.c_int
    P = ctypes.POINTER
    sig = {
        "bpe_abi_version": ([], ci),
        "bpe_create": ([ci, P(vp)], ci),
        "bpe_destroy": ([vp], ci),
        "bpe_last_error": ([vp], ctypes.c_char_p),
        "bpe_load_stream": ([vp, vp, u64, vp, u64], ci),
        "bpe_load_ids": ([vp, vp, u64, vp, u64], ci),
        "bpe_stream_len": ([vp, P(u64)], ci),
        "bpe_read_stream": ([vp, vp, u64, P(u64)], ci),
        "bpe_get_stats": ([vp, vp, vp, u64, P(u64)], ci),
        "bpe_merge": ([vp, i32, i32, i32, P(u64)], ci),
        "bpe_train": ([vp, i32, i32, vp, vp, P(i32)], ci),
        "bpe_replay": ([vp, vp, i32], ci),
        "bpe_encode": ([vp, vp, u64, vp, u64, vp, i32, vp, vp, u64, P(u64)], ci),
        "bpe_encode_text_gpt4": ([vp, vp, u64, vp, i32, vp, vp, u64, P(u64)], ci),
        "bpe_encode_text_gpt4_special": ([vp, vp, u64, vp, i32, vp, vp, vp, vp, i32, vp, u64, P(u64)], ci),
        "bpe_encode_batch_gpt4": ([vp, vp, u64, u64, vp, i32, vp, vp, vp, vp, i32, vp, u64, P(u64), vp], ci),
        "bpe_encode_stats": ([vp, vp], ci),
        "bpe_get_timing": ([vp, P(Timing)], ci),
        "bpe_set_option": ([vp, ci, i64], ci),
        "bpe_debug_table": ([vp, vp, vp, u64, P(u64)], ci),
        "bpe_gpt4_tables": ([vp, vp, vp], ci),
        "bpe_split_gpt4": ([vp, vp, u64, vp, u64, P(u64)], ci),
        "bpe_decode": ([vp, vp, u64, vp, u64, vp, vp, ctypes.c_int32, vp, u64, P(u64), P(ctypes.c_int64)], ci),
        "bpe_load_text_gpt4": ([vp, vp, u64, P(u64)], ci),
        "bpe_set_stream": ([vp, vp], ci),
        "bpe_step_begin": ([vp, vp], ci),
        "bpe_step_table": ([vp, vp, i32, i32, i32], ci),
        "bpe_step_select": ([vp, vp, i32], ci),
        "bpe_step_merge": ([vp, vp, vp], ci),
        "bpe_step_apply": ([vp, vp], ci),
        "bpe_step_delta_len": ([vp, P(u64)], ci),
        "bpe_step_poll": ([vp, P(i32), P(i32)], ci),
        "bpe_step_result": ([vp, vp, vp, i32, P(i32)], ci),
        "bpe_xchg_create": ([vp, i32, i32, i32, vp], ci),
        "bpe_xchg_attach": ([vp, vp], ci),
        "bpe_xchg_detach": ([vp], ci),
        "bpe_xchg_probe": ([vp, i32, P(i32)], ci),
        "bpe_step_fused": ([vp, i32], ci),
    }
    for name, (args, res) in sig.items():
        fn = getattr(L, name)  # AttributeError here = header/library mismatch
        fn.argtypes, fn.restype = args, res
    if L.bpe_abi_version() != ABI_VERSION:
        raise EngineError(f"libb200bpe ABI {L.bpe_abi_version()} != expected {ABI_VERSION}")
    _lib = L
    return L


def _ptr(a):
    return None if a is None else ctypes.c_void_p(a.ctypes.data)


def _as_offsets(offs):
    if offs is None:
        return None, 0
    o = np.ascontiguousarray(offs, dtype=np.uint64)
    return o, int(o.size)


class Engine:
    """One handle = one GPU = device-side state of one tokenizer (stream + pair table)."""

    def __init__(self, device=None):
        self._lib = load_library()
        if device is None:
            device = int(os.environ.get("LOCAL_RANK", "0")) if os.environ.get("BPE_DEVICE") is None else int(os.environ["BPE_DEVICE"])
        h = ctypes.c_void_p()
        rc = self._lib.bpe_create(int(device), ctypes.byref(h))
        if rc != 0:
            raise EngineError(f"bpe_create(device={device}) failed ({rc}): {self._lib.bpe_last_error(None).decode()}")
        self._h = h
        self.device = int(device)
        if os.environ.get("BPE_SEG_FILTER"):           # BPE_OPT_SEG_FILTER for every engine of the process (0 off, 1 when sparse, 2 always)
            self.set_option(OPT_SEG_FILTER, int(os.environ["BPE_SEG_FILTER"]))
        if os.environ.get("BPE_HIST_KERNEL"):          # BPE_OPT_HIST_KERNEL for every engine of the process (0 auto, 1 packed, 2 hashed)
            self.set_option(OPT_HIST_KERNEL, int(os.environ["BPE_HIST_KERNEL"]))

    def close(self):
        if getattr(self, "_h", None):
            self._lib.bpe_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise EngineError(f"{what} failed ({rc}): {self._lib.bpe_last_error(self._h).decode()}")

    # ---- corpus ----
    def load_stream(self, data, offsets=None):
        b = np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else np.ascontiguousarray(data, dtype=np.uint8)
        o, k = _as_offsets(offsets)
        self._keep = (b, o)
        self._check(self._lib.bpe_load_stream(self._h, _ptr(b) if b.size else None, b.size, _ptr(o), k), "bpe_load_stream")

    def load_ids(self, ids, offsets=None):
        a = np.ascontiguousarray(ids, dtype=np.int32)
        o, k = _as_offsets(offsets)
        self._check(self._lib.bpe_load_ids(self._h, _ptr(a) if a.size else None, a.size, _ptr(o), k), "bpe_load_ids")

    def stream_len(self):
        n = ctypes.c_uint64()
        self._check(self._lib.bpe_stream_len(self._h, ctypes.byref(n)), "bpe_stream_len")
        return n.value

    def read_stream(self):
        n = self.stream_len()
        out = np.empty(max(n, 1), dtype=np.int32)
        got = ctypes.c_uint64()
        self._check(self._lib.bpe_read_stream(self._h, _ptr(out), out.size, ctypes.byref(got)), "bpe_read_stream")
        return out[: got.value]

    # ---- primitives ----
    def get_stats(self):
        """-> (pairs[k,2] int32, counts[k] int64) in first-occurrence (dict insertion) order."""
        cap = max(self.stream_len(), 1)
        pairs = np.empty((cap, 2), dtype=np.int32)
        counts = np.empty(cap, dtype=np.int64)
        n = ctypes.c_uint64()
        self._check(self._lib.bpe_get_stats(self._h, _ptr(pairs), _ptr(counts), cap, ctypes.byref(n)), "bpe_get_stats")
        return pairs[: n.value], counts[: n.value]

    def merge(self, a, b, idx):
        n = ctypes.c_uint64()
        self._check(self._lib.bpe_merge(self._h, int(a), int(b), int(idx), ctypes.byref(n)), "bpe_merge")
        return n.value

    def train(self, num_merges, first_idx=256):
        """-> (pairs[k,2], counts[k], n_done); n_done < num_merges means the stream ran out of pairs."""
        pairs = np.zeros((max(num_merges, 1), 2), dtype=np.int32)
        counts = np.zeros(max(num_merges, 1), dtype=np.int64)
        done = ctypes.c_int32()
        self._check(self._lib.bpe_train(self._h, int(num_merges), int(first_idx), _ptr(pairs), _ptr(counts),
                                        ctypes.byref(done)), "bpe_train")
        return pairs[: done.value], counts[: done.value], done.value

    def replay(self, merges):
        """Apply `merges` ([M,2] int32, rank order) to the freshly loaded byte stream; train(first_idx=256+M) then resumes."""
        m = np.ascontiguousarray(np.asarray(merges, dtype=np.int32).reshape(-1, 2))
        self._check(self._lib.bpe_replay(self._h, _ptr(m) if m.size else None, m.shape[0]), "bpe_replay")

    def encode(self, data, offsets, merges, byte_perm=None):
        """-> ids int32.  merges: [M,2] int32 in rank order (id of rank r = 256 + r)."""
        b = np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else np.ascontiguousarray(data, dtype=np.uint8)
        o, k = _as_offsets(offsets)
        m = np.ascontiguousarray(np.asarray(merges, dtype=np.int32).reshape(-1, 2))
        perm = None if byte_perm is None else np.ascontiguousarray(byte_perm, dtype=np.uint8)
        out = np.empty(max(b.size, 1), dtype=np.int32)
        n = ctypes.c_uint64()
        self._check(self._lib.bpe_encode(self._h, _ptr(b) if b.size else None, b.size, _ptr(o), k,
                                         _ptr(m) if m.size else None, m.shape[0], _ptr(perm), _ptr(out), out.size,
                                         ctypes.byref(n)), "bpe_encode")
        return out[: n.value]

    def decode(self, ids, vocab_bytes, vocab_start, vocab_len):
        """-> (bytes, -1), or (None, i) when ids[i] is not in the vocabulary.  vocab_*: the flat vocabulary of
        bpe_decode (include/b200bpe.h)."""
        a = np.ascontiguousarray(ids, dtype=np.int32)
        vb = np.ascontiguousarray(vocab_bytes, dtype=np.uint8)
        vs = np.ascontiguousarray(vocab_start, dtype=np.uint64)
        vl = np.ascontiguousarray(vocab_len, dtype=np.uint32)
        n, bad = ctypes.c_uint64(), ctypes.c_int64(-1)
        cap = int(a.size) * 4 + 64
        for _ in range(2):
            out = np.empty(cap, dtype=np.uint8)
            rc = self._lib.bpe_decode(self._h, _ptr(a) if a.size else None, a.size, _ptr(vb) if vb.size else None, vb.size,
                                      _ptr(vs) if vs.size else None, _ptr(vl) if vl.size else None, int(vl.size), _ptr(out), cap,
                                      ctypes.byref(n), ctypes.byref(bad))
            if rc == -2 and bad.value >= 0:      # BPE_ERR_ARG with a position: an id outside the vocabulary
                return None, int(bad.value)
            if rc == -4 and n.value > cap:       # BPE_ERR_CAPACITY: the exact size is known now
                cap = int(n.value)
                continue
            self._check(rc, "bpe_decode")
            return out[: n.value].tobytes(), -1
        raise EngineError("bpe_decode: capacity retry failed")

    SPECIAL_MAX, SPECIAL_MAX_BYTES = 64, 48      # limits of bpe_encode_text_gpt4_special

    def encode_text_gpt4(self, data, merges, byte_perm=None, out=None, specials=None):
        """-> ids int32 of utf-8 `data`: GPT-4 split + encode, both on the GPU (regex.py:111-121).
        specials: [(utf-8 bytes, id), ...] in the order of the special_tokens dict — their occurrences are found on the
        GPU as well and every part between them is encoded on its own (regex.py:152-163)."""
        self._ensure_gpt4_tables()
        b = np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else np.ascontiguousarray(data, dtype=np.uint8)
        m = np.ascontiguousarray(np.asarray(merges, dtype=np.int32).reshape(-1, 2))
        perm = None if byte_perm is None else np.ascontiguousarray(byte_perm, dtype=np.uint8)
        if out is None:
            out = np.empty(max(b.size, 1), dtype=np.int32)
        n = ctypes.c_uint64()
        if specials:
            blob = np.frombuffer(b"".join(t for t, _ in specials), dtype=np.uint8)
            offs = np.zeros(len(specials) + 1, dtype=np.uint32)
            np.cumsum([len(t) for t, _ in specials], out=offs[1:])
            ids = np.asarray([i for _, i in specials], dtype=np.int32)
            self._check(self._lib.bpe_encode_text_gpt4_special(
                self._h, _ptr(b) if b.size else None, b.size, _ptr(m) if m.size else None, m.shape[0], _ptr(perm),
                _ptr(blob), _ptr(offs), _ptr(ids), len(specials), _ptr(out), out.size, ctypes.byref(n)), "bpe_encode_text_gpt4_special")
            return out[: n.value]
        self._check(self._lib.bpe_encode_text_gpt4(self._h, _ptr(b) if b.size else None, b.size, _ptr(m) if m.size else None,
                                                   m.shape[0], _ptr(perm), _ptr(out), out.size, ctypes.byref(n)), "bpe_encode_text_gpt4")
        return out[: n.value]

    def encode_batch_gpt4(self, data, n_docs, merges, byte_perm=None, specials=None):
        """-> (ids int32, doc_offsets int64[n_docs + 1]): the n_docs documents of `data` (their utf-8 joined by single 0xFF
        bytes) each split (BPE_OPT_SPLIT_PATTERN), special-token-cut and encoded on its own, all in one call; document d is
        ids[doc_offsets[d]:doc_offsets[d + 1]].  specials as in encode_text_gpt4."""
        self._ensure_gpt4_tables()
        b = np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else np.ascontiguousarray(data, dtype=np.uint8)
        m = np.ascontiguousarray(np.asarray(merges, dtype=np.int32).reshape(-1, 2))
        perm = None if byte_perm is None else np.ascontiguousarray(byte_perm, dtype=np.uint8)
        out = np.empty(max(b.size, 1), dtype=np.int32)          # every id covers at least one byte; separators give none
        doc = np.zeros(int(n_docs) + 1, dtype=np.uint64)
        blob, offs, ids, k = None, None, None, 0
        if specials:
            blob = np.frombuffer(b"".join(t for t, _ in specials), dtype=np.uint8)
            offs = np.zeros(len(specials) + 1, dtype=np.uint32)
            np.cumsum([len(t) for t, _ in specials], out=offs[1:])
            ids = np.asarray([i for _, i in specials], dtype=np.int32)
            k = len(specials)
        n = ctypes.c_uint64()
        self._check(self._lib.bpe_encode_batch_gpt4(
            self._h, _ptr(b) if b.size else None, b.size, int(n_docs), _ptr(m) if m.size else None, m.shape[0], _ptr(perm),
            _ptr(blob), _ptr(offs), _ptr(ids), k, _ptr(out), out.size, ctypes.byref(n), _ptr(doc)), "bpe_encode_batch_gpt4")
        return out[: n.value], doc.astype(np.int64)

    def encode_stats(self):
        a = np.zeros(10, dtype=np.uint64)
        self._check(self._lib.bpe_encode_stats(self._h, _ptr(a)), "bpe_encode_stats")
        names = ("memo_chunks", "pool_ids", "new_chunks", "direct_chunks", "long_chunks", "pieces", "fallback_pieces", "kernel_us",
                 "repeated_pieces", "direct_ids")
        return {k: int(v) for k, v in zip(names, a)}

    # ---- measurement / options ----
    def timing(self):
        t = Timing()
        self._check(self._lib.bpe_get_timing(self._h, ctypes.byref(t)), "bpe_get_timing")
        return t.as_dict()

    def set_option(self, opt, value):
        self._check(self._lib.bpe_set_option(self._h, int(opt), int(value)), "bpe_set_option")

    def debug_table(self):
        """Live entries of the incremental pair table: dict pair -> count (test hook)."""
        cap = 1 << 16
        while True:
            pairs = np.empty((cap, 2), dtype=np.int32)
            counts = np.empty(cap, dtype=np.int64)
            n = ctypes.c_uint64()
            rc = self._lib.bpe_debug_table(self._h, _ptr(pairs), _ptr(counts), cap, ctypes.byref(n))
            if rc == ERR_CAPACITY:
                cap = int(n.value) + 16
                continue
            self._check(rc, "bpe_debug_table")
            return {(int(p[0]), int(p[1])): int(c) for p, c in zip(pairs[: n.value], counts[: n.value])}

    # ---- GPT-4 split pattern on the device ----
    def _ensure_gpt4_tables(self):
        if not getattr(self, "_gpt4_ready", False):
            from .unicode_tables import tables
            cls, contr = tables()
            self._check(self._lib.bpe_gpt4_tables(self._h, _ptr(cls), _ptr(contr)), "bpe_gpt4_tables")
            self._gpt4_ready = True

    def split_gpt4(self, data):
        """Chunk start offsets (uint64) of utf-8 `data` under GPT4_SPLIT_PATTERN, computed on the GPU."""
        self._ensure_gpt4_tables()
        b = np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else np.ascontiguousarray(data, dtype=np.uint8)
        out = np.empty(max(b.size, 1), dtype=np.uint64)
        n = ctypes.c_uint64()
        self._check(self._lib.bpe_split_gpt4(self._h, _ptr(b) if b.size else None, b.size, _ptr(out), out.size, ctypes.byref(n)),
                    "bpe_split_gpt4")
        return out[: n.value].copy()

    def load_text_gpt4(self, data, count_chunks=False):
        """Upload utf-8 `data`, split it with GPT4_SPLIT_PATTERN on the GPU and make it the current stream."""
        self._ensure_gpt4_tables()
        b = np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else np.ascontiguousarray(data, dtype=np.uint8)
        n = ctypes.c_uint64()
        self._check(self._lib.bpe_load_text_gpt4(self._h, _ptr(b) if b.size else None, b.size,
                                                 ctypes.byref(n) if count_chunks else None), "bpe_load_text_gpt4")
        return n.value if count_chunks else None

    # ---- step-wise training (sharded loop; device pointers, e.g. torch tensors' data_ptr()) ----
    def set_stream(self, cuda_stream_ptr):
        self._check(self._lib.bpe_set_stream(self._h, ctypes.c_void_p(cuda_stream_ptr)), "bpe_set_stream")

    def step_begin(self, dense_ptr):
        self._check(self._lib.bpe_step_begin(self._h, ctypes.c_void_p(dense_ptr)), "bpe_step_begin")

    def step_table(self, dense_ptr, num_merges, first_idx=256, poll_every=16):
        self._check(self._lib.bpe_step_table(self._h, ctypes.c_void_p(dense_ptr), int(num_merges), int(first_idx),
                                             int(poll_every)), "bpe_step_table")

    def step_delta_len(self):
        n = ctypes.c_uint64()
        self._check(self._lib.bpe_step_delta_len(self._h, ctypes.byref(n)), "bpe_step_delta_len")
        return n.value

    def step_select(self, cand_ptr, rank):
        self._check(self._lib.bpe_step_select(self._h, ctypes.c_void_p(cand_ptr), int(rank)), "bpe_step_select")

    def step_merge(self, cand_ptr, delta_ptr):
        self._check(self._lib.bpe_step_merge(self._h, ctypes.c_void_p(cand_ptr), ctypes.c_void_p(delta_ptr)), "bpe_step_merge")

    def step_apply(self, delta_ptr):
        self._check(self._lib.bpe_step_apply(self._h, ctypes.c_void_p(delta_ptr)), "bpe_step_apply")

    def xchg_create(self, world, rank, vocab_cap):
        """Allocate this rank's NVLink exchange block; -> its 64-byte CUDA IPC handle (uint8 array)."""
        out = np.zeros(64, dtype=np.uint8)
        self._check(self._lib.bpe_xchg_create(self._h, int(world), int(rank), int(vocab_cap), _ptr(out)), "bpe_xchg_create")
        return out

    def xchg_attach(self, all_handles):
        a = np.ascontiguousarray(all_handles, dtype=np.uint8).reshape(-1)
        self._check(self._lib.bpe_xchg_attach(self._h, _ptr(a)), "bpe_xchg_attach")

    def xchg_probe(self, timeout_ms=3000):
        ok = ctypes.c_int32()
        self._check(self._lib.bpe_xchg_probe(self._h, int(timeout_ms), ctypes.byref(ok)), "bpe_xchg_probe")
        return bool(ok.value)

    def xchg_detach(self):
        self._check(self._lib.bpe_xchg_detach(self._h), "bpe_xchg_detach")

    def step_fused(self, n_iters):
        self._check(self._lib.bpe_step_fused(self._h, int(n_iters)), "bpe_step_fused")

    def step_poll(self):
        it, ex = ctypes.c_int32(), ctypes.c_int32()
        self._check(self._lib.bpe_step_poll(self._h, ctypes.byref(it), ctypes.byref(ex)), "bpe_step_poll")
        return it.value, bool(ex.value)

    def step_result(self, cap):
        pairs = np.zeros((max(cap, 1), 2), dtype=np.int32)
        counts = np.zeros(max(cap, 1), dtype=np.int64)
        done = ctypes.c_int32()
        self._check(self._lib.bpe_step_result(self._h, _ptr(pairs), _ptr(counts), int(cap), ctypes.byref(done)), "bpe_step_result")
        return pairs[: done.value], counts[: done.value], done.value
