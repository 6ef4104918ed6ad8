/*
 * b200bpe.h — C ABI of libb200bpe.so, the B200 (sm_100a) BPE train/encode hot path.
 *
 * The reference (karpathy/minbpe @1acefe8) is pure Python and has no FFI; its hot path is
 * the three primitives in minbpe/base.py plus the loops in basic.py / regex.py that drive
 * them.  Every entry point below names the reference lines it replaces.  The Python host
 * classes in minbpe_b200/tokenizer.py (same names and signatures as minbpe's Tokenizer /
 * BasicTokenizer / RegexTokenizer) call these through ctypes; INTEGRATION.md shows the stub
 * a minbpe maintainer would add to bind them.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / CUDA types cross the boundary.  Pointers are
 *     HOST pointers unless a parameter is named *_dev (a CUDA device pointer in the handle's
 *     device, for callers that keep buffers in HBM, e.g. torch.distributed all-reduce glue).
 *   - every function returns 0 (BPE_OK) or a negative bpe_status; bpe_last_error() gives the
 *     message.  Nothing throws across the ABI.  No global state besides per-handle state.
 *   - one handle = one GPU = one host thread at a time.  ctypes releases the GIL during calls.
 *   - token ids are int32 (the stream is held as 32-bit words in HBM; bit 31 is used
 *     internally as the "first token of a chunk" mark, so ids must be < 2^31).
 *   - a "stream" is the token sequence of the whole corpus plus chunk starts.  No pair and no
 *     merge ever crosses a chunk start (regex.py:51-54,60).  BasicTokenizer = one chunk.
 */
#ifndef B200BPE_H
#define B200BPE_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct bpe_handle bpe_handle;

typedef enum {
    BPE_OK = 0,
    BPE_ERR_CUDA = -1,      /* a CUDA runtime call failed (no device, OOM, launch error) */
    BPE_ERR_ARG = -2,       /* bad argument (NULL, out of range, unsorted offsets) */
    BPE_ERR_STATE = -3,     /* call order (e.g. train before load_stream) */
    BPE_ERR_CAPACITY = -4,  /* caller buffer too small; required size is reported */
    BPE_ERR_INTERNAL = -5
} bpe_status;

/* ---- lifetime ------------------------------------------------------------------------ */

/* Create a handle bound to CUDA device `device`.  Fails with BPE_ERR_CUDA when there is no
 * usable sm_100 device: there is NO CPU fallback.  (Stands where the reference constructs a
 * Tokenizer, base.py:69-74 — the handle is the device-side state of one tokenizer.) */
int bpe_create(int device, bpe_handle **out);
int bpe_destroy(bpe_handle *h);
/* Message for the last failing call on this handle ("" if none).  h may be NULL for a
 * failed bpe_create. */
const char *bpe_last_error(const bpe_handle *h);
/* ABI version of the loaded library (checked by the Python loader). */
int bpe_abi_version(void);

/* ---- loading a corpus into HBM --------------------------------------------------------- */

/* basic.py:25-26 (`ids = list(text.encode("utf-8"))`) and regex.py:41-44 (`findall` +
 * per-chunk `list(ch.encode("utf-8"))`): upload `n` text bytes and widen them to the int32
 * stream in HBM.  chunk_offsets[k] is the byte offset where chunk k starts (strictly
 * increasing, chunk_offsets[0] == 0); NULL / n_chunks==0 means one chunk (BasicTokenizer). */
int bpe_load_stream(bpe_handle *h, const uint8_t *bytes, uint64_t n,
                    const uint64_t *chunk_offsets, uint64_t n_chunks);

/* Same, for an arbitrary id list (what base.py:13 get_stats / base.py:25 merge accept). */
int bpe_load_ids(bpe_handle *h, const int32_t *ids, uint64_t n,
                 const uint64_t *chunk_offsets, uint64_t n_chunks);

/* Current stream length in tokens. */
int bpe_stream_len(bpe_handle *h, uint64_t *n);
/* Copy the current stream (ids only, chunk marks stripped) to out[0..cap).  *n = length;
 * BPE_ERR_CAPACITY if cap < *n. */
int bpe_read_stream(bpe_handle *h, int32_t *out, uint64_t cap, uint64_t *n);

/* ---- the three primitives -------------------------------------------------------------- */

/* base.py:13-22 get_stats(ids): adjacent-pair histogram of the loaded stream, overlaps
 * counted.  Results in dict insertion order, i.e. sorted by first occurrence in the stream:
 * pairs[2*i], pairs[2*i+1], counts[i].  *n_pairs = number of distinct pairs;
 * BPE_ERR_CAPACITY if cap < *n_pairs (call again with a larger buffer). */
int bpe_get_stats(bpe_handle *h, int32_t *pairs, int64_t *counts, uint64_t cap, uint64_t *n_pairs);

/* base.py:25-41 merge(ids, pair, idx): replace every left-to-right non-overlapping occurrence
 * of (a, b) in the loaded stream by idx.  *new_len = resulting stream length. */
int bpe_merge(bpe_handle *h, int32_t a, int32_t b, int32_t idx, uint64_t *new_len);

/* ---- the training loop ----------------------------------------------------------------- */

/* basic.py:31-45 / regex.py:49-66: run up to num_merges iterations of
 *     stats = get_stats(stream); pair = max(stats, key=stats.get); stream = merge(stream, pair, first_idx+i)
 * on the loaded stream, entirely on the device.  Ties are broken like the reference: among
 * the pairs with the highest count, the one whose first occurrence in the current stream is
 * earliest (dict insertion order, basic.py:35).
 *   out_pairs[2*i], out_pairs[2*i+1] : pair merged at iteration i (new id first_idx + i)
 *   out_counts[i]                    : stats[pair] before the merge (the number verbose mode
 *                                      prints, basic.py:45)
 *   *n_done                          : iterations completed.  n_done < num_merges means the
 *                                      stream ran out of pairs, where the reference raises
 *                                      ValueError (max() of an empty dict, basic.py:35); the
 *                                      call still returns BPE_OK. */
int bpe_train(bpe_handle *h, int32_t num_merges, int32_t first_idx,
              int32_t *out_pairs, int64_t *out_counts, int32_t *n_done);

/* Resume (base.py:140-165 load(), then more training): bring the freshly loaded BYTE stream (bpe_load_stream /
 * bpe_load_text_gpt4) to the state a training run has after the given merges — they are applied in rank order with
 * the training kernels, the pair table is maintained on the way — so that
 *     bpe_train(h, more, 256 + n_merges, ...)
 * continues that run: train(N) == train(k) -> save -> load -> bpe_replay(k merges) -> bpe_train(N - k). */
int bpe_replay(bpe_handle *h, const int32_t *merges, int32_t n_merges);

/* ---- encode ------------------------------------------------------------------------------ */

/* regex.py:92-121 (_encode_chunk per chunk, concatenated: encode_ordinary) and basic.py:57-74
 * (one chunk): for every chunk, repeatedly merge the present pair with the lowest merge rank.
 *   merges[2*r], merges[2*r+1] : pair of rank r; its id is 256 + r (base.py:159-165 order)
 *   byte_perm                  : NULL, or 256 entries mapping a text byte to its initial id
 *                                (gpt4.py:76-77,90-92)
 *   out_ids / out_cap / *out_n : caller buffer; n tokens always suffice.
 * Does not disturb a stream loaded for training. */
int bpe_encode(bpe_handle *h, const uint8_t *bytes, uint64_t n,
               const uint64_t *chunk_offsets, uint64_t n_chunks,
               const int32_t *merges, int32_t n_merges, const uint8_t *byte_perm,
               int32_t *out_ids, uint64_t out_cap, uint64_t *out_n);

/* regex.py:111-121 (encode_ordinary) with the GPT-4 split done on the device as well: text bytes in, ids out; no
 * chunk offsets exist anywhere (needs bpe_gpt4_tables).  Any length (pieces of 1 GiB cut at letter+space).
 * Every DISTINCT chunk is encoded once (k_encode2.cuh): the memo table and the rank table stay with the handle while
 * the caller keeps passing the same merges / byte_perm, so later calls and later pieces start warm.  bpe_encode with
 * chunk_offsets (any split pattern, offsets from the host) runs the same kernels. */
int bpe_encode_text_gpt4(bpe_handle *h, const uint8_t *bytes, uint64_t n, const int32_t *merges, int32_t n_merges,
                         const uint8_t *byte_perm, int32_t *out_ids, uint64_t out_cap, uint64_t *out_n);

/* RegexTokenizer.encode(text, allowed_special) — regex.py:123-164 — in one call.  The reference splits the text with
 * re.split("(" + "|".join(re.escape(k) for k in special) + ")", text) (leftmost match; the first special in dict order
 * that matches at a position wins; matches do not overlap), emits special[part] for every special and
 * encode_ordinary(part) for every part in between.  Here the occurrences are found on the device, become boundaries
 * of the GPT-4 split (the text on either side is split on its own) and single-id entries of the encode memo.
 * special_bytes: the specials' utf-8 bytes back to back, in dict order; special_offsets[n_special + 1]; at most 64
 * specials of 1..48 bytes each (BPE_ERR_ARG otherwise: the caller keeps the host split for those). */
int bpe_encode_text_gpt4_special(bpe_handle *h, const uint8_t *bytes, uint64_t n, const int32_t *merges, int32_t n_merges,
                                 const uint8_t *byte_perm, const uint8_t *special_bytes, const uint32_t *special_offsets,
                                 const int32_t *special_ids, int32_t n_special, int32_t *out_ids, uint64_t out_cap,
                                 uint64_t *out_n);
/* [tok.encode(t, allowed_special) for t in docs] in one call (regex.py:123-164 per document).  bytes = the n_docs documents'
 * UTF-8 joined by single 0xFF bytes (a byte UTF-8 never contains); every document is split (BPE_OPT_SPLIT_PATTERN) and
 * special-token-cut on its own.  Specials as in bpe_encode_text_gpt4_special (n_special = 0: none).  out_doc_offsets[n_docs + 1]:
 * document d's ids are out_ids[out_doc_offsets[d] .. out_doc_offsets[d + 1]).  BPE_ERR_ARG if bytes does not hold exactly
 * n_docs - 1 separators. */
int bpe_encode_batch_gpt4(bpe_handle *h, const uint8_t *bytes, uint64_t n, uint64_t n_docs,
                          const int32_t *merges, int32_t n_merges, const uint8_t *byte_perm,
                          const uint8_t *special_bytes, const uint32_t *special_offsets, const int32_t *special_ids,
                          int32_t n_special, int32_t *out_ids, uint64_t out_cap, uint64_t *out_n,
                          uint64_t *out_doc_offsets);
/* Counters of the memoised encode: out[0] distinct chunks in the memo table, [1] ids in its pool; of the last call:
 * [2] chunks newly added, [3] chunks encoded directly (no room in the table, or longer than 48 bytes), [4] of which
 * long, [5] pieces, [6] pieces that took the general path, [7] device microseconds of the encode kernels
 * (BPE_OPT_KERNEL_TIMING), [8] pieces done twice because the per-piece id area had to grow, [9] ids of the directly
 * encoded chunks of the last piece. */
int bpe_encode_stats(bpe_handle *h, uint64_t *out /* [10] */);

/* ---- the GPT-4 split pattern on the device (regex.py:19, used at regex.py:41 and :114) -------- */
/* `re.findall(GPT4_SPLIT_PATTERN, text)` as scans + element-wise kernels (k_split.cuh; the rules are
 * pinned against the `regex` module by tests/test_split_rules.py).  The caller provides the Unicode
 * class table of the regex engine it wants to match (minbpe_b200/unicode_tables.py enumerates the
 * installed `regex` module): cls_table[cp] in {0 letter, 1 number, 2 CR/LF, 3 other whitespace,
 * 4 apostrophe, 5 other} for cp < 0x110000, contr_table[cp] (cp < 0x3000) = bit0 (?i:[sdmt]),
 * bit1 (?i:l), bit2 (?i:v), bit3 (?i:e), bit4 (?i:r). */
int bpe_gpt4_tables(bpe_handle *h, const uint8_t *cls_table, const uint8_t *contr_table);
/* Chunk start offsets (bytes) of valid UTF-8 `bytes` under the GPT-4 pattern.  Any length: texts beyond 1 GiB are
 * processed in pieces cut at provable chunk boundaries (ASCII letter followed by U+0020). */
int bpe_split_gpt4(bpe_handle *h, const uint8_t *bytes, uint64_t n, uint64_t *out_offsets, uint64_t cap,
                   uint64_t *n_chunks);
/* regex.py:41-44 without the host: upload + split + widen; same stream as
 * bpe_load_stream(bytes, n, <offsets of the regex chunks>).  n_chunks may be NULL. */
int bpe_load_text_gpt4(bpe_handle *h, const uint8_t *bytes, uint64_t n, uint64_t *n_chunks);

/* ---- step-wise training: the sharded (multi-GPU) loop ---------------------------------------- */
/* One process per GPU, each holding a contiguous shard of the corpus (cut at chunk starts) and an
 * identical copy of the global pair-count table.  Per merge the host (minbpe_b200/dist.py) issues
 * two small collectives between these calls — MIN over one int64 (first-occurrence tie-break:
 * lowest rank = earliest text wins, basic.py:35 semantics across shards) and SUM over the
 * statistics delta vector — e.g. with torch.distributed / NCCL over NVLink.  *_dev parameters are
 * device pointers on the handle's GPU.  All work is enqueued on the stream set by bpe_set_stream
 * (the caller's stream, so its collectives are ordered with these kernels); nothing blocks the
 * host except bpe_step_table / bpe_step_poll / bpe_step_result. */
int bpe_set_stream(bpe_handle *h, void *cuda_stream /* cudaStream_t, NULL = the handle's own */);
/* regex.py:51-54 at iteration 0 on this shard: dense_dev[p0*256+p1] = local count (65536 uint64). */
int bpe_step_begin(bpe_handle *h, uint64_t *dense_dev);
/* Build the table from the all-reduced vector; prepare num_merges iterations with new ids from
 * first_idx.  poll_every = how many merges the host will enqueue between two bpe_step_poll calls. */
int bpe_step_table(bpe_handle *h, const uint64_t *dense_dev, int32_t num_merges, int32_t first_idx, int32_t poll_every);
/* regex.py:56 max(stats, key=stats.get): cand_dev[0] = rank << 58 | p0 << 29 | p1 for this rank's
 * candidate (global max count; on a tie the pair that occurs first in this shard), INT64_MAX if
 * this rank has none.  The host reduces cand_dev[0] with MIN across ranks. */
int bpe_step_select(bpe_handle *h, int64_t *cand_dev, int32_t rank);
/* regex.py:60 merge of the reduced winner in this shard; the statistics delta (DESIGN.md) is added
 * into delta_dev (uint64[bpe_step_delta_len], all zero on entry).  The host reduces it with SUM. */
int bpe_step_merge(bpe_handle *h, const int64_t *cand_dev, uint64_t *delta_dev);
/* Apply the summed delta to the table; zeroes delta_dev. */
int bpe_step_apply(bpe_handle *h, uint64_t *delta_dev);
int bpe_step_delta_len(bpe_handle *h, uint64_t *len);
/* Host sync: merges completed, whether the corpus ran out of pairs (reference: ValueError). */
int bpe_step_poll(bpe_handle *h, int32_t *iters_done, int32_t *exhausted);
/* Pairs and (global) counts of the merges performed so far. */
int bpe_step_result(bpe_handle *h, int32_t *out_pairs, int64_t *out_counts, int32_t cap, int32_t *n_done);

/* decode (basic.py:51-55, regex.py:78-90): out = vocab[ids[0]] + vocab[ids[1]] + ...  The vocabulary is
 * passed flat: vocab_bytes (all token bytes back to back), vocab_start[V] and vocab_len[V] per id;
 * vocab_len[id] = 0xffffffff marks an id that is not in the vocabulary.  *out_n = number of bytes (also
 * set when BPE_ERR_CAPACITY is returned, so the caller can size the buffer and call again).  An id that
 * is negative, >= V or marked absent ends the call with BPE_ERR_ARG and *bad_index = its position (the
 * reference raises ValueError in RegexTokenizer.decode, KeyError in BasicTokenizer.decode). */
int bpe_decode(bpe_handle *h, const int32_t *ids, uint64_t n_ids, const uint8_t *vocab_bytes, uint64_t vocab_nbytes,
               const uint64_t *vocab_start, const uint32_t *vocab_len, int32_t V, uint8_t *out, uint64_t cap,
               uint64_t *out_n, int64_t *bad_index);

/* ---- the same loop with the per-merge exchanges over NVLink peer memory (k_xchg.cuh) ------------- */
/* Replaces the two host-issued collectives per merge (MIN over the candidate, SUM over the delta vector) by
 * kernels that push / pull through CUDA-IPC-mapped peer memory: a tie pushes one candidate word to every
 * peer (a unique arg-max needs no exchange: the table is replicated), and the delta all-reduce is fused
 * with the table update (every rank pulls and sums the N local vectors while applying them).  No host call
 * per merge.  Sequence:
 *     bpe_xchg_create (every rank)  ->  all-gather the 64-byte handles (host)  ->  bpe_xchg_attach
 *     bpe_step_begin, all-reduce of the 65536-bin histogram (once), bpe_step_table         (as above)
 *     bpe_step_fused(n) ... bpe_step_poll ... bpe_step_result
 * vocab_cap must equal first_idx + num_merges of bpe_step_table.  world <= 16, one process per GPU on one
 * NVLink box (peer access required).  world == 1 works without peers and without CUDA IPC (the handle is zeroed). */
int bpe_xchg_create(bpe_handle *h, int32_t world, int32_t rank, int32_t vocab_cap, uint8_t *ipc_handle_out /* [64] */);
int bpe_xchg_attach(bpe_handle *h, const uint8_t *all_handles /* [world][64], own slot ignored */);
/* Handshake over the mapped blocks (every rank calls it): push a flag to every peer, wait for theirs, pull a magic
 * word from every peer; *ok = 1 when all of that worked within timeout_ms.  The host falls back to collectives otherwise. */
int bpe_xchg_probe(bpe_handle *h, int32_t timeout_ms, int32_t *ok);
/* Unmap the peers' blocks (before any rank re-creates or destroys its own: detach everywhere, synchronise the
 * ranks, then bpe_xchg_create / bpe_destroy). */
int bpe_xchg_detach(bpe_handle *h);
/* regex.py:49-63, n_iters iterations enqueued on the handle's stream; returns at once. */
int bpe_step_fused(bpe_handle *h, int32_t n_iters);

/* ---- measurement --------------------------------------------------------------------------- */

typedef struct {
    double loop_ms;          /* device time of the last bpe_train merge loop (CUDA events) */
    double init_ms;          /* device time of the initial histogram + table build (bpe_train); of the
                                split kernels after bpe_split_gpt4 / bpe_load_text_gpt4 with
                                BPE_OPT_KERNEL_TIMING */
    double merge_kernel_ms;  /* summed device time of the fused merge kernel launches when
                                per-kernel timing is on (BPE_OPT_KERNEL_TIMING), else 0 */
    uint64_t tokens_in;      /* sum over iterations of the stream length before the merge */
    uint64_t tokens_out;     /* sum over iterations of the stream length after the merge */
    uint64_t kernel_launches;/* kernels launched by the last bpe_train / bpe_encode call */
    uint64_t table_slots;    /* capacity of the pair-count table */
    uint64_t table_used;     /* occupied slots */
    uint64_t h2d_bytes;      /* host->device bytes copied by the last load/encode call */
    uint64_t d2h_bytes;      /* device->host bytes copied by the last train/encode/read call */
    uint64_t hist_kernel;    /* byte-pair histogram kernel of the last bpe_train / bpe_step_begin on a byte stream:
                                1 = k_hist_dense_packed, 2 = k_hist_dense (BPE_OPT_HIST_KERNEL), 0 = k_hist_dense, the choice
                                still open (no large stream seen yet) */
    uint64_t filter_candidates; /* BPE_OPT_SEG_FILTER: segments the filtered merges of the last bpe_train had to look at ... */
    uint64_t filter_segments;   /* ... of this many (sum over those merges of the number of segments); 0 = filter not used */
} bpe_timing;
int bpe_get_timing(bpe_handle *h, bpe_timing *out);

/* Options (bpe_set_option): */
#define BPE_OPT_KERNEL_TIMING 1 /* 1: bracket each fused-merge launch with CUDA events */
#define BPE_OPT_RESCAN 2        /* 1: rebuild the histogram from the stream every iteration
                                   instead of maintaining it incrementally (verification) */
#define BPE_OPT_BATCH 3         /* max merge iterations enqueued per host synchronisation */
#define BPE_OPT_TABLE_LOG2 4    /* log2 of the pair-count table capacity (0 = automatic) */
#define BPE_OPT_VOCAB_CAP 6     /* bpe_train: size the per-merge statistics delta vector for at least this vocabulary
                                   (a training run split over several bpe_train calls then keeps one layout; bench: the
                                   vocab-100000 configuration timed over a window of its merges) */
#define BPE_OPT_ENC_MEMO_LOG2 7 /* test hook: log2 of the slots of the encode memo table (0 = default 22); drops the current table */
#define BPE_OPT_SPLIT_PIECE 5   /* test hook: bytes per piece of the device splitter (0 = default 1 GiB); texts longer than
                                   a piece are cut where a letter is followed by U+0020 (process-wide) */
#define BPE_OPT_SPLIT_PATTERN 8 /* which of the reference's two split patterns (regex.py:18-19) the *_gpt4 entry points apply:
                                   0 = GPT4_SPLIT_PATTERN (default), 1 = GPT2_SPLIT_PATTERN; per handle */
#define BPE_OPT_HIST_KERNEL 9   /* byte-pair histogram of iteration 0: 2 = k_hist_dense (default: the kernel that has run on B200s);
                                   1 = k_hist_dense_packed; 0 = k_hist_dense until the first stream of >= 8 Mi tokens, where
                                   k_hist_dense_packed is cross-checked and timed against it and adopted if equal and not slower */
#define BPE_OPT_SEG_FILTER 10   /* bpe_train: skip the segments a merge cannot touch (per-segment id signatures + candidate list,
                                   k_seg_filter.cuh): 0 = off (default), 1 = from the batch after merges have become sparse
                                   (fewer replacements per merge than a 32nd of the segments), 2 = always */
int bpe_set_option(bpe_handle *h, int opt, int64_t value);

/* Test hook: live entries (count > 0) of the incrementally maintained pair-count table, in no
 * particular order.  After k merges it must equal get_stats() of the current stream
 * (tests/test_gpu_parity.py checks exactly that against the oracle). */
int bpe_debug_table(bpe_handle *h, int32_t *pairs, int64_t *counts, uint64_t cap, uint64_t *n_pairs);

#ifdef __cplusplus
}
#endif
#endif /* B200BPE_H */
