// k_encode2.cuh — encode_ordinary (regex.py:111-121) at corpus scale: every DISTINCT chunk is encoded once.
//
// regex.py:118-120 calls _encode_chunk (regex.py:92-109) for every regex chunk, and the result is a pure function
// of the chunk's bytes.  Text repeats its chunks (a GiB of prose has ~2*10^8 chunks but only 10^4..10^6 distinct
// ones), so the merge loop itself is run once per distinct chunk and every occurrence is a table lookup:
//
//   k_enc_insert    every chunk of at most E2_LMAX bytes claims a slot of the MEMO table (open addressing, the
//                   64-bit tag is claimed with one atomicCAS, the winner stores the chunk's bytes in the slot);
//                   newly claimed slots go on a work list; longer chunks, and chunks the table has no room for, go
//                   on the DIRECT list by position
//   k_enc_distinct  one thread per new slot: _encode_chunk (lowest-rank pair first, regex.py:97-108) on the slot's
//                   bytes, ids into the id pool, slot <- (ntok, offset)
//   k_enc_direct    listed chunks: short ones one thread each, long ones one CTA each (shared memory), ids into the
//                   pool, (position -> ntok, offset) into a small position map
//   k_enc_count     per 2 KiB tile of text: number of ids its chunks produce (lookup + EXACT compare of the
//                   chunk's bytes with the slot's, so a tag collision can never produce a wrong id: such a chunk
//                   is simply not found and falls to the position map / the failure flag)
//   (scan of the tile counts: k_flag_scan_parts)
//   k_enc_write     per tile: lookups again, ids staged in shared memory, coalesced stores to the output
//
// The memo table, the id pool and the rank table stay with the handle: further pieces of a long text, and later
// encode() calls with the same merges, start warm.
//
// HBM traffic per text byte: the text and its 1-byte chunk-start flags are read three times (insert, count,
// write) = 6 B, ids are written once (4 B per id, ~1.2 B per text byte); slots and pool entries of the hot
// chunks live in L2.  Algorithmic bytes (SURVEY.md §8d): 1 B read per text byte + 4 B written per id.
#pragma once
#include "common.cuh"
#include "k_encode.cuh"

#define E2_THREADS 256
#define E2_ITEMS 8
#define E2_TILE (E2_THREADS * E2_ITEMS)   // 2048 text bytes per CTA
#define E2_LMAX 48                        // chunks of up to 48 bytes are memoised (and encoded by one thread): key + header = one 64-byte slot
#define E2_KW (E2_LMAX / 4)               // key words
#define E2_PROBES 24
#define E2_HALO 64                        // bytes after the tile that its chunks may reach into (>= E2_LMAX + 4, multiple of 32)
#define E2_OUT (E2_TILE + E2_LMAX)           // ids of one tile staged in shared memory by k_enc_write
#define E2_PENDING 0xffu                  // MemoSlot.ntok while the slot has not been encoded yet
#define BATCH_SEP 0xffu                   // document separator of the batched encode (k_batch.cuh): a byte UTF-8 never contains

struct __align__(16) MemoSlot {           // 64 bytes
    u64 tag;                              // 0 = empty, else (hash | 1)
    u32 meta;                             // len (bits 0..7) | ntok (bits 8..15; E2_PENDING = not encoded yet)
    u32 off;                              // first id in the pool
    u32 key[E2_KW];                       // the chunk's bytes, zero padded
};
static_assert(sizeof(MemoSlot) == 64 && E2_LMAX % 16 == 0, "one slot = header + key = 64 bytes, key compared as 16-byte vectors");

#define E2_OFF_TMP 0x80000000u   // PosSlot.off / e2_resolve: the ids are in the per-piece area
struct __align__(16) PosSlot { u64 key; u32 ntok; u32 off; };   // key = chunk position + 1, 0 = empty

#define E2_FAIL_OTHER 1u                  // pool / lists full, an oversize chunk, a chunk nobody could resolve: general path
#define E2_FAIL_TMP 2u                    // the per-piece id area is too small: the host grows it and repeats the piece
struct EncCtl {
    ull memo_used;       // claimed memo slots
    ull pool_used;       // ids in the pool (encodings of memoised chunks: they live as long as the memo)
    u32 n_new;           // entries of the new-slot list
    u32 fail;            // E2_FAIL_* bits
    ull n_direct;        // entries of the direct list
    ull n_long;          // ... of which longer than E2_LMAX bytes
    ull tmp_used;        // ids in the per-piece area (encodings of the direct chunks of THIS piece)
};

struct Enc2 {
    const unsigned char *text;   // device text bytes
    const unsigned char *flag;   // 1 at every chunk start
    u64 n;
    MemoSlot *memo; u64 memo_mask; u64 memo_limit;
    u32 *pool; u64 pool_cap;
    u32 *tmp; u64 tmp_cap;           // per-piece id area; an offset with E2_OFF_TMP set points into it
    u32 *new_list; u32 new_cap;
    u64 *direct_list; u64 direct_cap;
    PosSlot *posmap; u64 pos_mask;
    EncCtl *ctl;
};

__device__ __forceinline__ u32 e2_id_at(const Enc2 &E, u32 off, u32 j) {
    return (off & E2_OFF_TMP) ? E.tmp[(off & ~E2_OFF_TMP) + j] : __ldg(&E.pool[off + j]);
}

// ---- a tile of text + chunk-start bits in shared memory -----------------------------------------------------
struct E2Tile {
    unsigned char *s_b;   // [E2_TILE + E2_HALO]
    u32 *s_bits;          // [(E2_TILE + E2_HALO) / 32]  bit p = a chunk starts at tile byte p (positions >= n count as starts)
};

__device__ __forceinline__ void e2_load_tile(const Enc2 &E, u64 lo, E2Tile T) {
    const u32 tid = threadIdx.x;
    // body: 8 bytes per thread
    {
        const u64 p = lo + (u64)tid * E2_ITEMS;
        uint2 tb = make_uint2(0, 0), fb = make_uint2(0x01010101u, 0x01010101u);
        if (p + E2_ITEMS <= E.n) {
            tb = *reinterpret_cast<const uint2 *>(E.text + p);
            fb = *reinterpret_cast<const uint2 *>(E.flag + p);
        } else {
            unsigned char t8[8], f8[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) { t8[k] = (p + k < E.n) ? E.text[p + k] : 0; f8[k] = (p + k < E.n) ? E.flag[p + k] : 1; }
            tb = make_uint2(t8[0] | (t8[1] << 8) | (t8[2] << 16) | ((u32)t8[3] << 24), t8[4] | (t8[5] << 8) | (t8[6] << 16) | ((u32)t8[7] << 24));
            fb = make_uint2(f8[0] | (f8[1] << 8) | (f8[2] << 16) | ((u32)f8[3] << 24), f8[4] | (f8[5] << 8) | (f8[6] << 16) | ((u32)f8[7] << 24));
        }
        *reinterpret_cast<uint2 *>(T.s_b + tid * E2_ITEMS) = tb;
        // 8 flag bytes (0/1) -> 8 bits
        u32 m = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) { m |= ((fb.x >> (8 * k)) & 1u) << k; m |= ((fb.y >> (8 * k)) & 1u) << (4 + k); }
        u32 w = m << (8 * (tid & 3));
        w |= __shfl_xor_sync(0xffffffffu, w, 1);
        w |= __shfl_xor_sync(0xffffffffu, w, 2);
        if ((tid & 3) == 0) T.s_bits[tid >> 2] = w;
    }
    // halo: E2_HALO bytes after the tile
    if (tid < E2_HALO) {
        const u64 p = lo + E2_TILE + tid;
        T.s_b[E2_TILE + tid] = (p < E.n) ? E.text[p] : 0;
        const u32 f = (p < E.n) ? E.flag[p] : 1u;
        const u32 w = __ballot_sync(0xffffffffu, f != 0);
        if ((tid & 31) == 0) T.s_bits[(E2_TILE >> 5) + (tid >> 5)] = w;
    }
    __syncthreads();
}

// length of the chunk starting at tile byte p: distance to the next start bit; E2_LMAX + 1 = "longer than E2_LMAX"
__device__ __forceinline__ u32 e2_chunk_len(const E2Tile &T, u32 p) {
    const u32 q = p + 1;
    const u32 wi = q >> 5, sh = q & 31u;
    const u64 two = ((u64)T.s_bits[wi] | ((u64)T.s_bits[wi + 1] << 32)) >> sh;     // start bits of bytes q .. q + 63 - sh
    u32 len;
    if (two) len = (u32)__ffsll((long long)two);
    else {                                                                          // ... and of the word after them
        const u32 third = T.s_bits[wi + 2];
        len = third ? (64u - sh) + (u32)__ffs(third) : E2_LMAX + 1;
    }
    return len > E2_LMAX ? E2_LMAX + 1 : len;
}

// 64-bit tag of a chunk from its zero-padded key words (never 0: bit 0 is set)
__device__ __forceinline__ u64 e2_tag(const u32 (&kw)[E2_KW], u32 len) {
    u64 h = 0x9e3779b97f4a7c15ull ^ ((u64)len << 56);
    h = hash64(h ^ ((u64)kw[0] | ((u64)kw[1] << 32)));
#pragma unroll
    for (u32 j = 2; j < E2_KW; j += 2)
        if (len > 4 * j) h = hash64(h ^ ((u64)kw[j] | ((u64)kw[j + 1] << 32)));
    return h | 1ull;
}

// key words of the chunk [p, p+len) of the tile (len <= E2_LMAX): zero padded; returns the tag
__device__ __forceinline__ u64 e2_key(const E2Tile &T, u32 p, u32 len, u32 (&kw)[E2_KW]) {
    const u32 *s32 = reinterpret_cast<const u32 *>(T.s_b);
    const u32 w0 = p >> 2, sh = (p & 3u) * 8u;
    const u32 nw = (len + 3u) >> 2;
#pragma unroll
    for (u32 j = 0; j < E2_KW; ++j) {
        u32 v = 0;
        if (j < nw) {
            v = __funnelshift_r(s32[w0 + j], s32[w0 + j + 1], sh);
            const u32 rem = len - 4u * j;
            if (rem < 4u) v &= (1u << (8u * rem)) - 1u;
        }
        kw[j] = v;
    }
    return e2_tag(kw, len);
}

__device__ __forceinline__ void e2_direct_append(const Enc2 &E, u64 pos, bool is_long) {
    const ull k = atomicAdd(&E.ctl->n_direct, 1ull);
    if (k < E.direct_cap) E.direct_list[k] = pos | (is_long ? (1ull << 63) : 0ull);
    else atomicOr(&E.ctl->fail, E2_FAIL_OTHER);
    if (is_long) atomicAdd(&E.ctl->n_long, 1ull);
}

// ---- pass 1: claim memo slots ------------------------------------------------------------------------------
// BATCH (k_batch.cuh): a chunk whose first byte is 0xFF is a document separator — never memoised, no ids, never a failure
template <bool BATCH>
__global__ void __launch_bounds__(E2_THREADS) k_enc_insert(Enc2 E) {
    __shared__ __align__(16) unsigned char s_b[E2_TILE + E2_HALO + 8];
    __shared__ u32 s_bits[(E2_TILE + E2_HALO) / 32 + 2];
    const E2Tile T{s_b, s_bits};
    const u64 lo = (u64)blockIdx.x * E2_TILE;
    if (threadIdx.x < 2) s_bits[(E2_TILE + E2_HALO) / 32 + threadIdx.x] = 0xffffffffu;
    e2_load_tile(E, lo, T);
    const u32 base = threadIdx.x * E2_ITEMS;
    u32 mine = (s_bits[base >> 5] >> (base & 31u)) & 0xffu;
    while (mine) {
        const u32 k = __ffs(mine) - 1;
        mine &= mine - 1;
        const u32 p = base + k;
        if (lo + p >= E.n) break;
        if (BATCH && s_b[p] == BATCH_SEP) continue;
        const u32 len = e2_chunk_len(T, p);
        if (len > E2_LMAX) { e2_direct_append(E, lo + p, true); continue; }
        u32 kw[E2_KW];
        const u64 tag = e2_key(T, p, len, kw);
        u64 slot = (tag >> 1) & E.memo_mask;
        bool placed = false;
#pragma unroll 1
        for (int probe = 0; probe < E2_PROBES; ++probe) {
            u64 t = ld_volatile_u64(&E.memo[slot].tag);
            if (t == 0) {
                if (*(volatile ull *)&E.ctl->memo_used >= E.memo_limit) break;      // table is as full as it may get
                t = atomicCAS((ull *)&E.memo[slot].tag, 0ull, (ull)tag);
                if (t == 0) {                                                     // claimed: this thread fills the slot
                    MemoSlot *m = &E.memo[slot];
                    m->meta = len | (E2_PENDING << 8);
#pragma unroll
                    for (int j = 0; j < E2_KW; ++j) m->key[j] = kw[j];
                    atomicAdd(&E.ctl->memo_used, 1ull);
                    const u32 q = atomicAdd(&E.ctl->n_new, 1u);
                    if (q < E.new_cap) E.new_list[q] = (u32)slot; else atomicOr(&E.ctl->fail, E2_FAIL_OTHER);
                    placed = true;
                    break;
                }
            }
            if (t == tag) { placed = true; break; }   // someone holds this tag (bytes are compared in the later passes)
            slot = (slot + 1) & E.memo_mask;
        }
        if (!placed) e2_direct_append(E, lo + p, false);
    }
}

// Special tokens (regex.py:152-163) as memo entries: the occurrence of a special is one chunk (k_special.cuh) whose
// "encoding" is its single id.  One thread per special, on a freshly cleared table.
__global__ void k_enc_seed_specials(Enc2 E, const unsigned char *__restrict__ blob, const u32 *__restrict__ off,
                                    const int *__restrict__ ids, int k) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= k) return;
    const u32 lo = off[s], len = off[s + 1] - lo;      // 1 .. E2_LMAX (checked by the host)
    u32 kw[E2_KW];
#pragma unroll
    for (u32 j = 0; j < E2_KW; ++j) {
        u32 v = 0;
        for (u32 t = 0; t < 4; ++t) if (4 * j + t < len) v |= (u32)blob[lo + 4 * j + t] << (8 * t);
        kw[j] = v;
    }
    const u64 tag = e2_tag(kw, len);
    u64 slot = (tag >> 1) & E.memo_mask;
    for (u64 probe = 0; probe <= E.memo_mask; ++probe) {
        const u64 old = atomicCAS((ull *)&E.memo[slot].tag, 0ull, (ull)tag);
        if (old == 0) {
            MemoSlot *m = &E.memo[slot];
            const ull o = atomicAdd(&E.ctl->pool_used, 1ull);
            if (o >= E.pool_cap) { atomicOr(&E.ctl->fail, E2_FAIL_OTHER); return; }
            E.pool[o] = (u32)ids[s];
            m->off = (u32)o;
#pragma unroll
            for (int j = 0; j < E2_KW; ++j) m->key[j] = kw[j];
            m->meta = len | (1u << 8);
            atomicAdd(&E.ctl->memo_used, 1ull);
            return;
        }
        slot = (slot + 1) & E.memo_mask;
    }
    atomicOr(&E.ctl->fail, E2_FAIL_OTHER);
}

// regex.py:92-109 on a short token list held by one thread.  tok[] in/out, returns the new length.
__device__ __forceinline__ u32 e2_encode_short(u32 *tok, u32 len, const RankTable &rt) {
    while (len >= 2) {
        u32 best = RANK_NONE, ba = 0, bb = 0;
        for (u32 i = 0; i + 1 < len; ++i) {
            const u32 r = rank_of(rt, tok[i], tok[i + 1]);
            if (r < best) { best = r; ba = tok[i]; bb = tok[i + 1]; }
        }
        if (best == RANK_NONE) break;
        const u32 z = 256u + best;
        u32 j = 0;
        for (u32 i = 0; i < len;) {
            if (i + 1 < len && tok[i] == ba && tok[i + 1] == bb) { tok[j++] = z; i += 2; }
            else tok[j++] = tok[i++];
        }
        len = j;
    }
    return len;
}

// ---- pass 2: encode every newly claimed slot once ------------------------------------------------------------
__global__ void __launch_bounds__(128) k_enc_distinct(Enc2 E, RankTable rt, const unsigned char *__restrict__ perm) {
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    const u32 n_new = min(E.ctl->n_new, E.new_cap);
    if (i >= n_new) return;
    MemoSlot *m = &E.memo[E.new_list[i]];
    const u32 len0 = m->meta & 0xffu;
    u32 tok[E2_LMAX];
    for (u32 k = 0; k < len0; ++k) {
        const u32 b = (m->key[k >> 2] >> (8u * (k & 3u))) & 0xffu;
        tok[k] = perm ? perm[b] : b;
    }
    const u32 len = e2_encode_short(tok, len0, rt);
    const ull off = atomicAdd(&E.ctl->pool_used, (ull)len);
    if (off + len > E.pool_cap) { atomicOr(&E.ctl->fail, E2_FAIL_OTHER); return; }
    for (u32 k = 0; k < len; ++k) E.pool[off + k] = tok[k];
    m->off = (u32)off;
    __threadfence();
    m->meta = len0 | (len << 8);
}

__device__ __forceinline__ void e2_pos_insert(const Enc2 &E, u64 pos, u32 ntok, u32 off) {
    const u64 key = pos + 1;
    u64 slot = hash64(key) & E.pos_mask;
    for (;;) {
        const u64 old = atomicCAS((ull *)&E.posmap[slot].key, 0ull, (ull)key);
        if (old == 0) { E.posmap[slot].ntok = ntok; E.posmap[slot].off = off; return; }
        slot = (slot + 1) & E.pos_mask;
    }
}

// ---- pass 3a: listed SHORT chunks (no room in the memo): one thread each --------------------------------------
__global__ void __launch_bounds__(128) k_enc_direct_short(Enc2 E, RankTable rt, const unsigned char *__restrict__ perm) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    const u64 nd = min((u64)E.ctl->n_direct, E.direct_cap);
    if (i >= nd) return;
    const u64 ent = E.direct_list[i];
    if (ent >> 63) return;
    const u64 pos = ent;
    u32 tok[E2_LMAX];
    u32 len0 = 0;
    for (u64 q = pos; q < E.n && len0 < E2_LMAX; ++q) {
        if (q > pos && E.flag[q]) break;
        const u32 b = E.text[q];
        tok[len0++] = perm ? perm[b] : b;
    }
    const u32 len = e2_encode_short(tok, len0, rt);
    const ull off = atomicAdd(&E.ctl->tmp_used, (ull)len);
    if (off + len > E.tmp_cap) { atomicOr(&E.ctl->fail, E2_FAIL_TMP); return; }
    for (u32 k = 0; k < len; ++k) E.tmp[off + k] = tok[k];
    e2_pos_insert(E, pos, len, (u32)off | E2_OFF_TMP);
}

// ---- pass 3b: listed LONG chunks: one CTA each, tokens in shared memory (as k_encode_long) --------------------
__global__ void __launch_bounds__(256) k_enc_direct_long(Enc2 E, RankTable rt, const unsigned char *__restrict__ perm) {
    extern __shared__ u32 sm[];
    u32 *tk = sm, *tk2 = sm + ENC_LONG_MAX;
    __shared__ u32 s_scan[256];
    __shared__ u32 s_best, s_a, s_b2, s_len, s_len0;
    __shared__ ull s_off;
    const u32 tid = threadIdx.x;
    const u64 nd = min((u64)E.ctl->n_direct, E.direct_cap);
    for (u64 q = blockIdx.x; q < nd; q += gridDim.x) {
        const u64 ent = E.direct_list[q];
        if (!(ent >> 63)) continue;                       // block-uniform
        const u64 pos = ent & ~(1ull << 63);
        // chunk end: next start flag (the first E2_LMAX bytes hold none)
        if (tid == 0) s_len0 = 0xffffffffu;
        __syncthreads();
        for (u64 base = pos + 1; ; base += 256) {
            const u64 p = base + tid;
            const bool hit = (p >= E.n) || E.flag[p];
            if (hit) atomicMin(&s_len0, (u32)min(p - pos, (u64)0xfffffffeu));
            __syncthreads();
            if (s_len0 != 0xffffffffu || base - pos > ENC_LONG_MAX) break;
            __syncthreads();
        }
        __syncthreads();
        const u32 len0 = s_len0;
        if (len0 > ENC_LONG_MAX) { if (tid == 0) atomicOr(&E.ctl->fail, E2_FAIL_OTHER); __syncthreads(); continue; }   // host: general path
        for (u32 i = tid; i < len0; i += 256) { const u32 b = E.text[pos + i]; tk[i] = perm ? perm[b] : b; }
        u32 len = len0;
        __syncthreads();
        for (;;) {
            if (len < 2) break;
            if (tid == 0) s_best = RANK_NONE;
            __syncthreads();
            u32 best = RANK_NONE;
            for (u32 i = tid; i + 1 < len; i += 256) { const u32 r = rank_of(rt, tk[i], tk[i + 1]); best = r < best ? r : best; }
            if (best != RANK_NONE) atomicMin(&s_best, best);
            __syncthreads();
            best = s_best;
            if (best == RANK_NONE) break;
            for (u32 i = tid; i + 1 < len; i += 256)
                if (rank_of(rt, tk[i], tk[i + 1]) == best) { s_a = tk[i]; s_b2 = tk[i + 1]; }
            __syncthreads();
            const u32 a = s_a, b = s_b2, z = 256u + best;
            if (a != b) {
                for (u32 i = tid; i < len; i += 256) {
                    const bool st = (i + 1 < len) && tk[i] == a && tk[i + 1] == b;
                    const bool tail = (i >= 1) && tk[i - 1] == a && tk[i] == b;
                    tk2[i] = st ? 1u : (tail ? 2u : 0u);
                }
            } else if (tid == 0) {
                for (u32 i = 0; i < len;) {
                    if (i + 1 < len && tk[i] == a && tk[i + 1] == a) { tk2[i] = 1u; tk2[i + 1] = 2u; i += 2; }
                    else { tk2[i] = 0u; i += 1; }
                }
            }
            __syncthreads();
            const u32 per = (len + 255) / 256;
            const u32 s0 = min(len, tid * per), s1 = min(len, s0 + per);
            u32 kept = 0;
            for (u32 i = s0; i < s1; ++i) kept += (tk2[i] != 2u);
            s_scan[tid] = kept;
            __syncthreads();
            for (int o = 1; o < 256; o <<= 1) {
                const u32 v = (tid >= (u32)o) ? s_scan[tid - o] : 0;
                __syncthreads();
                s_scan[tid] += v;
                __syncthreads();
            }
            const u32 dst = s_scan[tid] - kept;
            if (tid == 255) s_len = s_scan[255];
            __syncthreads();
            u32 outv[32];
            u32 m = 0;
            for (u32 i = s0; i < s1; ++i) {
                const u32 f = tk2[i];
                if (f != 2u) outv[m++] = (f == 1u) ? z : tk[i];
            }
            __syncthreads();
            for (u32 k = 0; k < m; ++k) tk2[dst + k] = outv[k];
            __syncthreads();
            len = s_len;
            for (u32 i = tid; i < len; i += 256) tk[i] = tk2[i];
            __syncthreads();
        }
        __syncthreads();
        if (tid == 0) s_off = atomicAdd(&E.ctl->tmp_used, (ull)len);
        __syncthreads();
        const ull off = s_off;
        if (off + len > E.tmp_cap) { if (tid == 0) atomicOr(&E.ctl->fail, E2_FAIL_TMP); }
        else {
            for (u32 i = tid; i < len; i += 256) E.tmp[off + i] = tk[i];
            if (tid == 0) e2_pos_insert(E, pos, len, (u32)off | E2_OFF_TMP);
        }
        __syncthreads();
    }
}

// ---- lookup: (ntok, offset) of the chunk at tile byte p ------------------------------------------------------
__device__ __forceinline__ bool e2_resolve(const Enc2 &E, const E2Tile &T, u64 lo, u32 p, u32 &ntok, u32 &off) {
    const u32 len = e2_chunk_len(T, p);
    if (len <= E2_LMAX) {
        u32 kw[E2_KW];
        const u64 tag = e2_key(T, p, len, kw);
        u64 slot = (tag >> 1) & E.memo_mask;
#pragma unroll 1
        for (int probe = 0; probe < E2_PROBES; ++probe) {
            const MemoSlot *m = &E.memo[slot];
            const uint4 head = *reinterpret_cast<const uint4 *>(m);            // tag, meta, off
            const u64 t = (u64)head.x | ((u64)head.y << 32);
            if (t == 0) break;
            if (t == tag) {
                bool same = (head.z & 0xffu) == len;
#pragma unroll
                for (int v = 0; v < E2_KW / 4; ++v) {                           // the key, 16 bytes at a time
                    const uint4 k = *reinterpret_cast<const uint4 *>(m->key + 4 * v);
                    same = same && k.x == kw[4 * v] && k.y == kw[4 * v + 1] && k.z == kw[4 * v + 2] && k.w == kw[4 * v + 3];
                }
                const u32 nt = (head.z >> 8) & 0xffu;
                if (same && nt != E2_PENDING) { ntok = nt; off = head.w; return true; }
                break;   // a different chunk with the same tag (or a slot that could not be encoded): position map
            }
            slot = (slot + 1) & E.memo_mask;
        }
    }
    if (E.posmap) {
        const u64 key = lo + p + 1;
        u64 slot = hash64(key) & E.pos_mask;
        for (;;) {
            const u64 k = E.posmap[slot].key;
            if (k == key) { ntok = E.posmap[slot].ntok; off = E.posmap[slot].off; return true; }
            if (k == 0) break;
            slot = (slot + 1) & E.pos_mask;
        }
    }
    return false;
}

// ---- pass 4: ids per tile -------------------------------------------------------------------------------------
// BATCH: also the number of separators of the tile -> sep_part
template <bool BATCH>
__global__ void __launch_bounds__(E2_THREADS) k_enc_count(Enc2 E, u32 *__restrict__ part, u32 *__restrict__ sep_part) {
    __shared__ __align__(16) unsigned char s_b[E2_TILE + E2_HALO + 8];
    __shared__ u32 s_bits[(E2_TILE + E2_HALO) / 32 + 2];
    __shared__ u32 s_red[E2_THREADS / 32];
    __shared__ u32 s_red_sep[BATCH ? E2_THREADS / 32 : 1];
    const E2Tile T{s_b, s_bits};
    const u64 lo = (u64)blockIdx.x * E2_TILE;
    if (threadIdx.x < 2) s_bits[(E2_TILE + E2_HALO) / 32 + threadIdx.x] = 0xffffffffu;
    e2_load_tile(E, lo, T);
    const u32 base = threadIdx.x * E2_ITEMS;
    u32 mine = (s_bits[base >> 5] >> (base & 31u)) & 0xffu;
    u32 sum = 0, nsep = 0;
    while (mine) {
        const u32 k = __ffs(mine) - 1;
        mine &= mine - 1;
        const u32 p = base + k;
        if (lo + p >= E.n) break;
        if (BATCH && s_b[p] == BATCH_SEP) { ++nsep; continue; }
        u32 nt = 0, off = 0;
        if (e2_resolve(E, T, lo, p, nt, off)) sum += nt; else atomicOr(&E.ctl->fail, E2_FAIL_OTHER);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = sum;
    if (BATCH) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) nsep += __shfl_xor_sync(0xffffffffu, nsep, o);
        if ((threadIdx.x & 31) == 0) s_red_sep[threadIdx.x >> 5] = nsep;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        u32 t = 0;
        for (int w = 0; w < E2_THREADS / 32; ++w) t += s_red[w];
        part[blockIdx.x] = t;
        if (BATCH) {
            u32 c = 0;
            for (int w = 0; w < E2_THREADS / 32; ++w) c += s_red_sep[w];
            sep_part[blockIdx.x] = c;
        }
    }
}

// ---- pass 5: write the ids ------------------------------------------------------------------------------------
// BATCH: separator s of the piece (sep_excl[tile] + the separators in front of it in the tile) closes a document:
// doc_out[s] = out_base + its output position
template <bool BATCH>
__global__ void __launch_bounds__(E2_THREADS) k_enc_write(Enc2 E, const u64 *__restrict__ excl, int *__restrict__ out,
                                                          const u64 *__restrict__ sep_excl, u64 *__restrict__ doc_out, u64 out_base) {
    __shared__ __align__(16) unsigned char s_b[E2_TILE + E2_HALO + 8];
    __shared__ u32 s_bits[(E2_TILE + E2_HALO) / 32 + 2];
    __shared__ u32 s_scan[E2_THREADS / 32];
    __shared__ u32 s_scan_sep[BATCH ? E2_THREADS / 32 : 1];
    // ids of the tile's chunks in output order: the first E2_OUT of them are staged here and stored coalesced; a
    // long chunk that starts in this tile can carry more ids than the tile has bytes — those go straight to HBM
    __shared__ u32 s_out[E2_OUT];
    const E2Tile T{s_b, s_bits};
    const u64 lo = (u64)blockIdx.x * E2_TILE;
    if (threadIdx.x < 2) s_bits[(E2_TILE + E2_HALO) / 32 + threadIdx.x] = 0xffffffffu;
    e2_load_tile(E, lo, T);
    const u32 tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const u32 base = tid * E2_ITEMS;
    const u32 bits = (s_bits[base >> 5] >> (base & 31u)) & 0xffu;
    u32 nts[E2_ITEMS], offs[E2_ITEMS];
    u32 sum = 0, cnt = 0;
    u32 mine = bits;
    u32 sep_bits = 0, nsep = 0;     // BATCH: bit c = chunk c of this thread is a separator
    while (mine) {
        const u32 k = __ffs(mine) - 1;
        mine &= mine - 1;
        const u32 p = base + k;
        if (lo + p >= E.n) break;
        if (BATCH && s_b[p] == BATCH_SEP) { sep_bits |= 1u << cnt; ++nsep; nts[cnt] = 0; offs[cnt] = 0; ++cnt; continue; }
        u32 nt = 0, off = 0;
        e2_resolve(E, T, lo, p, nt, off);
        nts[cnt] = nt; offs[cnt] = off; ++cnt;
        sum += nt;
    }
    u32 incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const u32 v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= (u32)o) incl += v; }
    if (lane == 31) s_scan[warp] = incl;
    u32 sep_incl = 0;
    if constexpr (BATCH) {
        sep_incl = nsep;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const u32 v = __shfl_up_sync(0xffffffffu, sep_incl, o); if (lane >= (u32)o) sep_incl += v; }
        if (lane == 31) s_scan_sep[warp] = sep_incl;
    }
    __syncthreads();
    u32 wbase = 0, total = 0;
#pragma unroll
    for (int w = 0; w < E2_THREADS / 32; ++w) { const u32 v = s_scan[w]; if ((u32)w < warp) wbase += v; total += v; }
    u32 dst = wbase + incl - sum;
    int *o = out + excl[blockIdx.x];
    if constexpr (BATCH) if (sep_bits) {
        u64 s = sep_excl[blockIdx.x] + sep_incl - nsep;
#pragma unroll
        for (int w = 0; w < E2_THREADS / 32; ++w) if ((u32)w < warp) s += s_scan_sep[w];
        u32 d = dst;
        for (u32 c = 0; c < cnt; ++c) {
            if ((sep_bits >> c) & 1u) doc_out[s++] = out_base + excl[blockIdx.x] + d;
            d += nts[c];
        }
    }
    for (u32 c = 0; c < cnt; ++c) {
        const u32 nt = nts[c], off = offs[c];
        for (u32 j = 0; j < nt; ++j) {
            const u32 v = e2_id_at(E, off, j);
            if (dst + j < E2_OUT) s_out[dst + j] = v; else o[dst + j] = (int)v;
        }
        dst += nt;
    }
    __syncthreads();
    const u32 staged = total < E2_OUT ? total : E2_OUT;
    for (u32 i = tid; i < staged; i += E2_THREADS) o[i] = (int)s_out[i];
}

// chunk-start flags from host offsets (callers that bring their own split: bpe_encode with chunk_offsets)
__global__ void k_enc_flags_from_offsets(unsigned char *__restrict__ flag, const u64 *__restrict__ offs, u64 k, u64 n) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < k; i += (u64)gridDim.x * blockDim.x) {
        const u64 o = offs[i];
        if (o < n) flag[o] = 1;
    }
}
