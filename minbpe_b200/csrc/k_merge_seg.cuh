// k_merge_seg.cuh — the fused merge pass (base.py:25-41 + the statistics delta) for a != b on the
// SEGMENTED stream.  One WARP owns one 512-token segment at a time: 16 tokens per lane in
// registers, compacted in place, independently of every other segment.  There is no prefix sum
// across segments and no block-level synchronisation in the loop: every warp is its own pipeline.
//
//   read   4 * count bytes per segment        (one 1-D bulk async copy, TMA / UBLKCP, into the
//                                              warp's private mbarrier ring, MS_STAGES deep)
//   write  only from the 32-byte sector that holds the first changed word to the new end of the
//          segment (16-byte stores, same address range); nothing for an untouched segment
//   + 32-byte edge records per segment (first 3 / last 2 tokens, count), double-buffered, so a
//     warp can see across its segment boundaries without reading a body that another warp rewrites
//
// Work distribution: a ticket (one atomic) hands a warp MS_BATCH consecutive segments; the warp
// loads their edge records once, then keeps MS_STAGES-1 bulk copies in flight ahead of the segment
// it is working on.  The marking and delta rules are the ones documented in k_merge.cuh.
#pragma once
#include "common.cuh"
#include "k_merge.cuh"
#include "k_seg.cuh"

#ifndef MS_WARPS
#define MS_WARPS 8
#endif
#define MS_THREADS (MS_WARPS * 32)
#ifndef MS_STAGES
#define MS_STAGES 2
#endif
#ifndef MS_MINBLOCKS
#define MS_MINBLOCKS 4
#endif
#ifndef MS_DCACHE_LOG2
#define MS_DCACHE_LOG2 9
#endif
#ifndef MS_BATCH
#define MS_BATCH 8                          // consecutive segments per ticket
#endif
#define MS_PAD 4                            // body starts at word 4 of a stage (16-byte aligned); s[-1], s[-2] = previous tokens
#define MS_SW (SEG_TOKENS + 8)              // words per stage: pad, body, three following tokens
#define MS_META 16                          // per stage: P0 P1 N0 N1 N2 seg count - | the segment's own edge record
#define MS_BE (MS_BATCH + 2)                // edge records of a batch and of the segment on either side
#define MS_DCACHE (1 << MS_DCACHE_LOG2)     // slots of the per-CTA delta cache (shared memory)
#define MS_WARP_WORDS (MS_STAGES * MS_SW + MS_STAGES * MS_META + MS_BE * 8)
#define MS_SMEM_BYTES (MS_WARPS * MS_WARP_WORDS * 4 + MS_WARPS * MS_STAGES * 8 + MS_DCACHE * 8 + 16)
#define MS_INVALID 0xffffffffu
static_assert(SEG_TOKENS == 512, "k_merge_seg: a lane owns 4 rows x 4 tokens of a 512-token segment");
static_assert((MS_SW * 4) % 16 == 0 && (MS_WARP_WORDS * 4) % 16 == 0, "bulk-copy destinations must stay 16-byte aligned");

// delta[idx] += 1 through a CTA-private shared-memory cache: the same few neighbour ids are hit by
// almost every merge of a dense iteration (global same-address atomics serialise in L2); the
// persistent CTA folds them here and flushes once at exit.
__device__ __noinline__ void delta_cache_add(u32 *s_dkey, u32 *s_dcnt, ull *delta, u32 idx) {
    u32 slot = (idx * 2654435761u) >> (32 - MS_DCACHE_LOG2);
#pragma unroll 1
    for (int probe = 0; probe < 4; ++probe) {
        u32 k = reinterpret_cast<volatile u32 *>(s_dkey)[slot];
        if (k == 0xffffffffu) {
            const u32 old = atomicCAS(&s_dkey[slot], 0xffffffffu, idx);
            k = (old == 0xffffffffu) ? idx : old;
        }
        if (k == idx) { atomicAdd(&s_dcnt[slot], 1u); return; }
        slot = (slot + 1) & (MS_DCACHE - 1);
    }
    atomicAdd(&delta[idx], 1ull);   // cache neighbourhood full
}

// statistics delta of the merge that starts at the token at shared address `at` (rules: k_merge.cuh).
// The words at s[-2..-1] and s[count..count+2] hold the neighbouring segments' tokens (or the sentinel).
__device__ __noinline__ void delta_one(u32 at, u32 a, u32 b, u32 V, u32 *s_dkey, u32 *s_dcnt, ull *delta) {
    const u32 t0 = lds32(at), tm1 = lds32o<-4>(at), tm2 = lds32o<-8>(at), tp2 = lds32o<8>(at), tp3 = lds32o<12>(at);
    const bool m_m2 = (((tm2 ^ a) & TOK_MASK) == 0) && tm1 == b;   // a merge starts two tokens earlier
    const bool m_p2 = (((tp2 ^ a) & TOK_MASK) == 0) && tp3 == b;   // a merge starts two tokens later
    if (tm1 != TOK_SENTINEL && !(t0 & TOK_FLAG) && !m_m2) delta_cache_add(s_dkey, s_dcnt, delta, tm1 & TOK_MASK);
    if (!(tp2 & TOK_FLAG))   // also false for the sentinel (end of stream)
        delta_cache_add(s_dkey, s_dcnt, delta, m_p2 ? 2u * V : V + tp2);
}

struct SegArgs {
    Ctl *ctl;
    u32 *buf0, *buf1;
    Edge *e0, *e1;
    ull *delta;   // [0,V) L, [V,2V) R, [2V] ZZ; NULL = plain merge
    u32 V;
    int force;
    const unsigned char *xbase;   // sharded loop: the rank's exchange block (k_xchg.cuh); the delta vector is then
    u64 xstride;                  // the one of the current round's parity inside it, and `delta` is ignored
};

// one row (128 tokens, 4 per lane) into bits 4R..4R+3 of the lane's masks: m = merge starts (a at the token, b after it),
// pm = token 0 of the row follows an a (it is dropped if it is b).  Bits of tokens past the end of the segment are cleared
// by the valid mask.
template <int R>
__device__ __forceinline__ void mark_row(u32 la, u32 a, u32 b, u32 (&t)[4], u32 &m, u32 &pm) {
    const uint4 q = lds128o<R * 512>(la);
    const u32 nx = lds32o<R * 512 + 16>(la), pv = lds32o<R * 512 - 4>(la);
    t[0] = q.x; t[1] = q.y; t[2] = q.z; t[3] = q.w;
    m |= (((t[0] ^ a) & TOK_MASK) == 0 && t[1] == b) ? (1u << (4 * R)) : 0u;
    m |= (((t[1] ^ a) & TOK_MASK) == 0 && t[2] == b) ? (2u << (4 * R)) : 0u;
    m |= (((t[2] ^ a) & TOK_MASK) == 0 && t[3] == b) ? (4u << (4 * R)) : 0u;
    m |= (((t[3] ^ a) & TOK_MASK) == 0 && nx == b) ? (8u << (4 * R)) : 0u;
    pm |= (((pv ^ a) & TOK_MASK) == 0 && t[0] == b) ? (1u << (4 * R)) : 0u;
}

// the merged token takes the place of the merge start (bit 4R+i of mn) in the registers
template <int R>
__device__ __forceinline__ void replace_row(u32 mn, u32 z, u32 (&t)[4]) {
    if (mn & (1u << (4 * R))) t[0] = z | (t[0] & TOK_FLAG);
    if (mn & (2u << (4 * R))) t[1] = z | (t[1] & TOK_FLAG);
    if (mn & (4u << (4 * R))) t[2] = z | (t[2] & TOK_FLAG);
    if (mn & (8u << (4 * R))) t[3] = z | (t[3] & TOK_FLAG);
}

// write the kept tokens of one row to their compacted place (word offset `off` of the stage)
__device__ __forceinline__ void scatter_row(u32 s_a, u32 lane, u32 off, u32 row_kept, u32 lane_excl, u32 kp, const u32 (&t)[4]) {
    if (row_kept == 128u) {                 // warp-uniform: nothing dropped in this row, it only moves
        const u32 p = s_a + ((off + 4u * lane) << 2);
        if ((off & 3u) == 0) sts128(p, t[0], t[1], t[2], t[3]);
        else { sts32(p, t[0]); sts32o<4>(p, t[1]); sts32o<8>(p, t[2]); sts32o<12>(p, t[3]); }
    } else {
        u32 p = s_a + ((off + lane_excl) << 2);
        if (kp & 1u) sts32(p, t[0]);
        p += (kp << 2) & 4u;
        if (kp & 2u) sts32(p, t[1]);
        p += (kp << 1) & 4u;
        if (kp & 4u) sts32(p, t[2]);
        p += kp & 4u;
        if (kp & 8u) sts32(p, t[3]);
    }
}

// LIST = false: every segment of the stream, MS_BATCH consecutive ones per ticket.  LIST = true: only the candidate segments
// k_seg_filter put on the list at ctl->cand_ptr, one per ticket (the filter carried the other segments' edge records over).
template <bool LIST>
__global__ void __launch_bounds__(MS_THREADS, MS_MINBLOCKS) k_merge_seg(SegArgs A) {
    Ctl *ctl = A.ctl;
    if (!A.force && (ctl->done || ctl->overflow || ctl->iter >= ctl->max_iter)) return;
    if (ctl->a == ctl->b) return;  // pairs (a,a) take the pack + k_merge<true> path

    extern __shared__ __align__(128) unsigned char smem_raw[];
    u32 *s_warp = reinterpret_cast<u32 *>(smem_raw);                              // [MS_WARPS][MS_WARP_WORDS]
    u64 *s_bar = reinterpret_cast<u64 *>(s_warp + MS_WARPS * MS_WARP_WORDS);      // [MS_WARPS][MS_STAGES]
    u32 *s_dkey = reinterpret_cast<u32 *>(s_bar + MS_WARPS * MS_STAGES);          // [MS_DCACHE] delta index or 0xffffffff
    u32 *s_dcnt = s_dkey + MS_DCACHE;                                             // [MS_DCACHE]
    ull *s_drops = reinterpret_cast<ull *>(s_dcnt + MS_DCACHE);

    const u32 FULL = 0xffffffffu;
    const u32 tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const u64 n = ctl->n;
    u32 *__restrict__ w = ctl->cur ? A.buf1 : A.buf0;                 // compacted in place
    const Edge *__restrict__ e_cur = ctl->edge_cur ? A.e1 : A.e0;
    Edge *__restrict__ e_next = ctl->edge_cur ? A.e0 : A.e1;
    const u32 a = (u32)ctl->a, b = (u32)ctl->b, z = (u32)ctl->z;
    const u32 nseg = ctl->nseg;
    ull *const delta = A.xbase ? x_local_delta(A.xbase, A.xstride) : A.delta;
    const u32 *__restrict__ cand = LIST ? reinterpret_cast<const u32 *>(ctl->cand_ptr) : nullptr;
    const u32 n_cand = LIST ? ctl->n_cand : 0u;

    // this warp's private shared memory, as 32-bit shared-window byte addresses
    const u32 ws_a = smem_addr(s_warp + warp * MS_WARP_WORDS);   // [MS_STAGES][MS_SW] staging ring
    const u32 wmeta_a = ws_a + MS_STAGES * MS_SW * 4;            // [MS_STAGES][MS_META]
    const u32 wbe_a = wmeta_a + MS_STAGES * MS_META * 4;         // [MS_BE][8] edge records batch_seg-1 .. batch_seg+MS_BATCH
    const u32 wbar_a = smem_addr(s_bar + warp * MS_STAGES);

    if (lane == 0) {
        for (int s = 0; s < MS_STAGES; ++s) mbar_init(s_bar + warp * MS_STAGES + s, 1);
        fence_mbar_init();
    }
    for (u32 i = tid; i < MS_DCACHE; i += MS_THREADS) { s_dkey[i] = 0xffffffffu; s_dcnt[i] = 0; }
    if (tid == 0) *s_drops = 0;
    __syncthreads();

    // ---- issue side: next non-empty segment of this warp -> bulk copy into `stage` ----
    u32 batch_seg = 0, batch_pos = MS_BATCH;   // warp-uniform
    u32 list_next = blockIdx.x * MS_WARPS + warp;   // LIST: this warp's next entry of the candidate list
    // byte offset inside the batch's edge-record window (relative to record k) of the word lane l copies
    // into meta[l]: meta[0..4] = P0 P1 N0 N1 N2 = previous record's l[1], l[0], next record's f[0..2];
    // meta[8..15] = the segment's own record (for the untouched case); meta[5] = seg, meta[6] = count
    const u32 meta_src = 4u * (lane == 0 ? 4u : lane == 1 ? 3u : lane < 5 ? 14u + lane : lane < 8 ? 0u : lane < 16 ? lane : 0u);
    bool exhausted = false;
    auto issue = [&](u32 stage) {
        const u32 meta_a = wmeta_a + stage * (MS_META * 4);
        for (;;) {
            if (exhausted) {
                if (lane == 0) sts32o<20>(meta_a, MS_INVALID);
                __syncwarp();
                return;
            }
            if (batch_pos == MS_BATCH) {
                u32 tk = 0;
                if (LIST) {
                    // one candidate at a time, list entries dealt out round-robin over all warps of the grid (a ticket per
                    // entry would be one atomic on one address per segment); its record and its neighbours' go to the last
                    // three slots of the window, where the code below finds those of the last segment of a batch
                    tk = list_next; list_next += gridDim.x * MS_WARPS;
                    if (tk >= n_cand) { exhausted = true; continue; }
                    batch_seg = cand[tk] - (MS_BATCH - 1); batch_pos = MS_BATCH - 1;
                } else {
                    if (lane == 0) tk = atomicAdd(&ctl->merge_ticket, 1u);
                    tk = __shfl_sync(FULL, tk, 0);
                    if ((u64)tk * MS_BATCH >= nseg) { exhausted = true; continue; }
                    batch_seg = tk * MS_BATCH; batch_pos = 0;
                }
                if (LIST ? (lane >= MS_BATCH - 1 && lane < MS_BE) : (lane < MS_BE)) {
                    const long long idx = (LIST ? (long long)(int)batch_seg : (long long)batch_seg) - 1 + lane;   // LIST: batch_seg may have wrapped below 0
                    uint4 q0, q1;   // f0 f1 f2 l0 | l1 count pad pad
                    if (idx >= 0 && idx < (long long)nseg) {
                        const uint4 *p = reinterpret_cast<const uint4 *>(&e_cur[idx]);
                        q0 = p[0]; q1 = p[1];
                    } else {        // past either end of the stream: a "long" neighbour made of sentinels
                        q0 = make_uint4(TOK_SENTINEL, TOK_SENTINEL, TOK_SENTINEL, TOK_SENTINEL);
                        q1 = make_uint4(TOK_SENTINEL, 3u, 0u, 0u);
                    }
                    sts128(wbe_a + lane * 32, q0.x, q0.y, q0.z, q0.w);
                    sts128(wbe_a + lane * 32 + 16, q1.x, q1.y, q1.z, q1.w);
                }
                __syncwarp();
            }
            const u32 k = batch_pos++;
            const u32 seg = batch_seg + k;
            if (seg >= nseg) { exhausted = true; continue; }
            const u32 rec_a = wbe_a + k * 32;          // record k = the segment in front of this one
            const u32 cnt = lds32o<32 + 20>(rec_a);
            if (cnt == 0) {   // empty segment: only its (empty) edge record is carried over
                if (lane < 8) reinterpret_cast<u32 *>(&e_next[seg])[lane] = (lane < 5) ? TOK_SENTINEL : 0u;
                continue;
            }
            const u32 cm1 = lds32o<20>(rec_a), cp1 = lds32o<64 + 20>(rec_a);
            const u32 st_a = ws_a + stage * (MS_SW * 4);
            u32 mv = lds32(rec_a + meta_src);
            if (lane == 5) mv = seg;
            if (lane == 6) mv = cnt;
            if (lane < 16) sts32(meta_a + lane * 4, mv);
            if (lane < 2) sts32(st_a + (MS_PAD - 1 - lane) * 4, mv);   // s[-1] = P0, s[-2] = P1
            if (!(cm1 >= 2 && cp1 >= 3)) {   // short / empty neighbours: walk the edge records
                __syncwarp();
                if (lane == 0) {
                    u32 N[3], P[2];
                    seg_neighbours(e_cur, seg, nseg, N, P);
                    sts32o<0>(meta_a, P[0]); sts32o<4>(meta_a, P[1]); sts32o<8>(meta_a, N[0]); sts32o<12>(meta_a, N[1]); sts32o<16>(meta_a, N[2]);
                    sts32o<(MS_PAD - 1) * 4>(st_a, P[0]); sts32o<(MS_PAD - 2) * 4>(st_a, P[1]);
                }
            }
            __syncwarp();
            if (lane == 0) {
                const u32 bytes = ((cnt + 3u) & ~3u) * 4u;
                fence_proxy_async_smem();   // the stage was last written with ordinary stores (in-place compaction)
                mbar_arrive_expect_tx_a(wbar_a + stage * 8, bytes);
                bulk_g2s_a(st_a + MS_PAD * 4, w + (u64)seg * SEG_TOKENS, bytes, wbar_a + stage * 8);
            }
            __syncwarp();
            return;
        }
    };

    for (u32 s = 0; s + 1 < MS_STAGES; ++s) issue(s);
    u32 drops = 0;
    for (u32 j = 0;; ++j) {
        const u32 stage = j % MS_STAGES;
        issue((j + MS_STAGES - 1) % MS_STAGES);   // the stage consumed in the previous round
        const u32 meta_a = wmeta_a + stage * (MS_META * 4);
        const u32 seg = lds32o<20>(meta_a);
        if (seg == MS_INVALID) break;
        const u32 count = lds32o<24>(meta_a);
        const u32 s_a = ws_a + stage * (MS_SW * 4) + MS_PAD * 4;   // address of token 0 of the segment
        mbar_wait_a(wbar_a + stage * 8, (j / MS_STAGES) & 1u);
        if (lane < 3) sts32(s_a + (count + lane) * 4, lds32(meta_a + 8 + lane * 4));   // the three tokens that follow
        __syncwarp();

        // ---- mark: row r = tokens [128r, 128r+128), four consecutive tokens per lane.  A lane's 16 tokens are bits
        //      4r+i of its masks; in that order their stream positions 128r + 4*lane + i increase, so the tokens this
        //      segment owns (position < count) are a prefix of the bits ----
        u32 t[4][4], m = 0, pm = 0;
        const u32 la = s_a + lane * 16;
        mark_row<0>(la, a, b, t[0], m, pm);
        if (count > 128u) mark_row<1>(la, a, b, t[1], m, pm);   // short segments (the sparse end of training) skip rows
        if (count > 256u) mark_row<2>(la, a, b, t[2], m, pm);
        if (count > 384u) mark_row<3>(la, a, b, t[3], m, pm);
        const u32 nvalid = 4u * (count >> 7) + (u32)min(max((int)(count & 127u) - (int)(4u * lane), 0), 4);
        const u32 valid = (1u << nvalid) - 1u;
        const u32 mn = m & valid;                                  // a merge only starts at a token this segment owns
        const u32 keep = ~(((m << 1) & 0xeeeeu) | pm) & valid;     // dropped: the token after a merge start
        // lowest position whose word changes (a merge start or a dropped token); rows and words in front of it stay
        const u32 ch = mn | (keep ^ valid);
        const u32 cb = __ffs(ch) - 1u;
        const u32 first = ~__reduce_max_sync(FULL, ch ? ~((cb >> 2) * 128u + lane * 4u + (cb & 3u)) : 0u);   // MS_INVALID: none
        if (first == MS_INVALID) {
            // untouched segment: nothing to write, the edge record carries over
            if (lane < 8) reinterpret_cast<u32 *>(&e_next[seg])[lane] = lds32(meta_a + 32 + lane * 4);
            __syncwarp();
            continue;
        }

        // ---- statistics delta of this segment's merge starts (reads the stage before it is rewritten) ----
        if (delta) {
            u32 mall = mn;
#pragma unroll 1
            while (mall) {   // one pass per merge start of this lane
                const int bit = __ffs(mall) - 1;
                mall &= mall - 1;
                delta_one(la + (bit >> 2) * 512 + (bit & 3) * 4, a, b, A.V, s_dkey, s_dcnt, delta);
            }
        }

        if (mn) {   // few lanes
            replace_row<0>(mn, z, t[0]);
            replace_row<1>(mn, z, t[1]);
            replace_row<2>(mn, z, t[2]);
            replace_row<3>(mn, z, t[3]);
        }

        // ---- kept tokens per lane and row, packed one byte per row: one warp scan for all four rows ----
        const u32 own = __popc(keep & 0xfu) | (__popc(keep & 0xf0u) << 8) | (__popc(keep & 0xf00u) << 16) | (__popc(keep & 0xf000u) << 24);
        u32 incl = own;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const u32 v = __shfl_up_sync(FULL, incl, o);
            if (lane >= (u32)o) incl += v;          // a row keeps at most 128 tokens: no carry between bytes
        }
        const u32 tot = __shfl_sync(FULL, incl, 31);
        const u32 excl = incl - own;
        const u32 k0 = tot & 0xffu, k1 = (tot >> 8) & 0xffu, k2 = (tot >> 16) & 0xffu, k3 = tot >> 24;
        const u32 off1 = k0, off2 = k0 + k1, off3 = off2 + k2;
        const u32 new_count = off3 + k3;
        const u32 first_row = first >> 7;           // rows in front of it stay where they are
        __syncwarp();                               // all lanes hold their tokens; delta reads are done

        // ---- compact in place inside the stage, from the first changed row on (a row past the end keeps nothing) ----
        if (first_row == 0) scatter_row(s_a, lane, 0u, k0, excl & 0xffu, keep & 0xfu, t[0]);
        if (first_row <= 1 && k1) scatter_row(s_a, lane, off1, k1, (excl >> 8) & 0xffu, (keep >> 4) & 0xfu, t[1]);
        if (first_row <= 2 && k2) scatter_row(s_a, lane, off2, k2, (excl >> 16) & 0xffu, (keep >> 8) & 0xfu, t[2]);
        if (k3) scatter_row(s_a, lane, off3, k3, excl >> 24, keep >> 12, t[3]);
        __syncwarp();
        // ---- copy-out: 16-byte vectors from the 32-byte sector that holds the first changed word to the new end (the
        //      up to three words past new_count land in the dead part of the segment) ----
        {
            uint4 *__restrict__ gp = reinterpret_cast<uint4 *>(w + (u64)seg * SEG_TOKENS) + lane;
            const u32 vend = (new_count + 3u) >> 2, vbeg = (first >> 3) * 2u;
            if (lane >= vbeg && lane < vend) gp[0] = lds128o<0>(la);
            if (lane + 32u >= vbeg && lane + 32u < vend) gp[32] = lds128o<512>(la);
            if (lane + 64u >= vbeg && lane + 64u < vend) gp[64] = lds128o<1024>(la);
            if (lane + 96u >= vbeg && lane + 96u < vend) gp[96] = lds128o<1536>(la);
        }
        // ---- the segment's new edge record ----
        {
            // lane:  0 1 2 -> f[0..2]   3 4 -> l[0], l[1] = tokens new_count-2, new_count-1   5 -> count   6 7 -> 0
            const u32 idx = lane < 3 ? lane : new_count + lane - 5u;
            const bool have = lane < 3 ? (lane < new_count) : (new_count + lane >= 5u);
            u32 word = TOK_SENTINEL;
            if (have && lane < 5) word = lds32(s_a + (idx & (SEG_TOKENS - 1)) * 4);
            if (lane == 5) word = new_count;
            if (lane > 5) word = 0;
            if (lane < 8) reinterpret_cast<u32 *>(&e_next[seg])[lane] = word;   // Edge = f[3], l[2], count, pad[2]
        }
        drops += count - new_count;
        __syncwarp();   // the stage may be refilled from here on
    }

    if (lane == 0 && drops) atomicAdd(s_drops, (ull)drops);
    __syncthreads();
    if (delta)
        for (u32 i = tid; i < MS_DCACHE; i += MS_THREADS)
            if (s_dkey[i] != 0xffffffffu && s_dcnt[i]) atomicAdd(&delta[s_dkey[i]], (ull)s_dcnt[i]);
    // ---- exit: the last CTA out publishes the new stream length and flips the edge arrays ----
    if (tid == 0) {
        const ull cta_drops = *s_drops;
        if (cta_drops) atomicAdd(&ctl->drops, cta_drops);
        __threadfence();
        const u32 e = atomicAdd(&ctl->merge_exit, 1u);
        if (e == gridDim.x - 1) {
            __threadfence();
            const ull dropped = *(volatile ull *)&ctl->drops;
            ctl->sum_in += n; ctl->sum_out += n - dropped;
            ctl->n = n - dropped;
            ctl->drops = 0;
            ctl->edge_cur ^= 1u;
            ctl->iter += 1;
            ctl->epoch += 1;
            ctl->merge_ticket = 0; ctl->merge_exit = 0;
        }
    }
}
