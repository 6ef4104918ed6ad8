// b200bpe.cu — host side of libb200bpe.so: the C ABI of include/b200bpe.h over the sm_100a
// kernels in k_load.cuh / k_stats.cuh / k_merge.cuh / k_encode.cuh.
//
// Build: see build.py (nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -shared).
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "../../include/b200bpe.h"
#include "common.cuh"
#include "k_load.cuh"
#include "k_merge.cuh"
#include "k_merge_seg.cuh"
#include "k_seg.cuh"
#include "k_seg_filter.cuh"
#include "k_stats.cuh"
#include "k_encode.cuh"
#include "k_split.cuh"
#include "k_decode.cuh"
#include "k_xchg.cuh"
#include "k_encode2.cuh"
#include "k_special.cuh"
#include "k_batch.cuh"

#define BPE_ABI_VERSION 1

struct EncState;
struct SpecSet;
struct GenEnc;
struct bpe_handle {
    int device = 0;
    EncState *enc = nullptr;          // memoised chunk encode (encode2_host.inl): rank table, memo, id pool, scratch
    bpe_handle *enc_scratch = nullptr;   // general encode path (encode_host.inl) works on its own stream buffers
    SpecSet *spec = nullptr;             // special tokens of the current encode call (special_host.inl)
    GenEnc *gen = nullptr;               // general encode path: device scratch + the rank table of the last merges seen (encode_host.inl)
    int sms = 0;
    cudaStream_t stream = nullptr;       // the stream every kernel of this handle runs on
    cudaStream_t own_stream = nullptr;   // created by bpe_create; `stream` may point at a caller's stream instead
    std::string err;

    // token stream: two ping-pong buffers of cap_tokens words
    u32 *buf[2] = {nullptr, nullptr};
    u64 cap_tokens = 0;
    bool loaded = false;
    bool bytes_only = false;  // every id < 256 (fresh byte stream)

    Ctl *ctl = nullptr;    // device
    Ctl *h_ctl = nullptr;  // pinned host mirror

    Table table = {nullptr, nullptr, nullptr, 0};
    bool table_valid = false;  // table == get_stats(current stream)
    u64 *desc = nullptr; u64 desc_cap = 0;
    Edge *edge[2] = {nullptr, nullptr}; u64 *seg_offs = nullptr; u64 seg_cap = 0;  // segmented stream metadata
    ull *delta = nullptr; u32 V = 0;   // V = layout of the delta vector the kernels index (L[0,V) R[V,2V) ZZ[2V])
    u32 delta_cap = 0;                 // vocabulary capacity of the OWNED buffer `delta` (step mode uses the caller's)
    u32 max_id = 255;                  // largest id in the loaded stream (bpe_load_ids); byte streams: 255
    ull *dense = nullptr;
    ull *dense2 = nullptr; u32 *d_cmp = nullptr;   // first-use cross-check of the packed histogram kernel (hist_dense)
    int hist_mode = 0;                             // 0 = not decided, 1 = k_hist_dense_packed, 2 = k_hist_dense
    // segment filter (k_seg_filter.cuh): signatures, candidate list
    u32 *sig = nullptr, *cand = nullptr; u64 sig_cap = 0;
    bool filt_active = false;                      // the iterations being enqueued use the filter
    bool sig_valid = false;                        // the signatures describe the current stream
    u32 *d_err = nullptr;
    int *log_pairs = nullptr; long long *log_counts = nullptr; int log_cap = 0;
    Best *partials = nullptr;
    unsigned char *d_cls = nullptr, *d_contr = nullptr;   // code-point class / contraction tables of the GPT-4 splitter
    // sharded loop over NVLink peer memory (k_xchg.cuh): the rank's exchange block and its peers' mappings
    unsigned char *xchg = nullptr; u64 xchg_bytes = 0, xchg_stride = 0; u32 xchg_V = 0;
    XArgs xargs = {};
    bool xchg_attached = false;
    u32 *d_present = nullptr;   // sharded loop: bitmap of pair hashes that have occurred in this shard (k_stats.cuh)
    unsigned char *split_slab = nullptr; u64 split_cap = 0;   // working set of the splitter, kept between calls (split_host.inl)
    int argmax_grid = 0, merge_grid_same = 0, merge_grid_seg = 0, ff_grid = 0;

    // options
    int step_poll_every = 16;
    int opt_kernel_timing = 0, opt_rescan = 0, opt_batch = 256, opt_table_log2 = 0;
    int opt_memo_log2 = 0;   // BPE_OPT_ENC_MEMO_LOG2 (test hook): log2 slots of the encode memo table, 0 = default
    u32 opt_vocab_cap = 0;   // BPE_OPT_VOCAB_CAP: lower bound of the delta-vector layout V used by bpe_train
    int opt_seg_filter = 0;      // BPE_OPT_SEG_FILTER: 0 = off, 1 = switch it on when merges have become sparse, 2 = always
    int opt_hist_kernel = 2;     // BPE_OPT_HIST_KERNEL: 2 = k_hist_dense (default: the kernel that has run on B200s), 1 = k_hist_dense_packed,
                                 // 0 = decide at the first large stream (cross-check + timing)
    int opt_split_pattern = 0;   // BPE_OPT_SPLIT_PATTERN: 0 = GPT-4 split pattern, 1 = GPT-2 (bpe_split_gpt4 / bpe_load_text_gpt4 / bpe_encode_text_gpt4*)

    bpe_timing tm = {};
    std::vector<cudaEvent_t> ev_pool;  // per-launch timing of the fused merge kernel (BPE_OPT_KERNEL_TIMING)
    int ev_used = 0;
};

static thread_local std::string g_create_err;
static void xchg_release(bpe_handle *h);
static void enc2_free(bpe_handle *h);
static void spec_free(bpe_handle *h);
static void gen_free(bpe_handle *h);
static u64 g_split_piece_override = 0;   // BPE_OPT_SPLIT_PIECE (test hook): bytes per piece of the device splitter

static int fail(bpe_handle *h, int code, const std::string &msg) {
    if (h) h->err = msg; else g_create_err = msg;
    return code;
}

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(h, BPE_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));      \
    } while (0)

static inline int grid_for(u64 work_items, int threads, int max_blocks) {
    u64 b = (work_items + threads - 1) / threads;
    if (b < 1) b = 1;
    if (b > (u64)max_blocks) b = max_blocks;
    return (int)b;
}

extern "C" int bpe_abi_version(void) { return BPE_ABI_VERSION; }

extern "C" const char *bpe_last_error(const bpe_handle *h) { return h ? h->err.c_str() : g_create_err.c_str(); }

// ------------------------------------------------------------------------------------------------
static int free_table(bpe_handle *h, Table &t) {
    if (t.keys) cudaFree(t.keys);
    if (t.counts) cudaFree(t.counts);
    if (t.first) cudaFree(t.first);
    t = {nullptr, nullptr, nullptr, 0};
    (void)h;
    return BPE_OK;
}

static int alloc_table(bpe_handle *h, Table &t, u64 cap, bool with_first) {
    t = {nullptr, nullptr, nullptr, cap - 1};
    CU(cudaMalloc(&t.keys, cap * 8));
    CU(cudaMalloc(&t.counts, cap * 8));
    if (with_first) CU(cudaMalloc(&t.first, cap * 8));
    CU(cudaMemsetAsync(t.keys, 0xff, cap * 8, h->stream));
    CU(cudaMemsetAsync(t.counts, 0, cap * 8, h->stream));
    if (with_first) CU(cudaMemsetAsync(t.first, 0xff, cap * 8, h->stream));
    return BPE_OK;
}

static u64 next_pow2(u64 x) { u64 p = 1; while (p < x) p <<= 1; return p; }

extern "C" int bpe_create(int device, bpe_handle **out) {
    bpe_handle *h = nullptr;
    if (!out) return fail(nullptr, BPE_ERR_ARG, "bpe_create: out is NULL");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, BPE_ERR_CUDA, std::string("bpe_create: no CUDA device (") + cudaGetErrorString(e) +
                                               "); libb200bpe has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(nullptr, BPE_ERR_ARG, "bpe_create: device index out of range");
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) return fail(nullptr, BPE_ERR_CUDA, cudaGetErrorString(e));
    if (prop.major != 10)
        return fail(nullptr, BPE_ERR_CUDA, std::string("bpe_create: device '") + prop.name + "' is sm_" +
                                               std::to_string(prop.major) + std::to_string(prop.minor) +
                                               "; this library contains sm_100a code only");
    h = new (std::nothrow) bpe_handle();
    if (!h) return fail(nullptr, BPE_ERR_INTERNAL, "out of host memory");
    h->device = device;
    h->sms = prop.multiProcessorCount;
    auto bail = [&](const char *what, cudaError_t ce) {
        std::string m = std::string(what) + ": " + cudaGetErrorString(ce);
        delete h;
        return fail(nullptr, BPE_ERR_CUDA, m);
    };
    if ((e = cudaSetDevice(device)) != cudaSuccess) return bail("cudaSetDevice", e);
    if ((e = cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking)) != cudaSuccess) return bail("cudaStreamCreate", e);
    h->stream = h->own_stream;
    if ((e = cudaMalloc(&h->ctl, sizeof(Ctl))) != cudaSuccess) return bail("cudaMalloc ctl", e);
    if ((e = cudaMallocHost(&h->h_ctl, sizeof(Ctl))) != cudaSuccess) return bail("cudaMallocHost", e);
    if ((e = cudaMalloc(&h->dense, 65536 * 8)) != cudaSuccess) return bail("cudaMalloc dense", e);
    if ((e = cudaMalloc(&h->d_err, 8)) != cudaSuccess) return bail("cudaMalloc err", e);   // [0] error flag, [1] max id seen by k_copy_ids
    int occ_same = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_same, k_merge<true>, MG_THREADS, 0);
    if (occ_same < 1) occ_same = 1;
    h->merge_grid_same = h->sms * occ_same;
    int occ_fast = 0;
    if ((e = cudaFuncSetAttribute(k_merge_seg<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, MS_SMEM_BYTES)) != cudaSuccess)
        return bail("cudaFuncSetAttribute(k_merge_seg)", e);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_fast, k_merge_seg<false>, MS_THREADS, MS_SMEM_BYTES);
    if (occ_fast < 1) return bail("k_merge_seg does not fit on an SM", cudaErrorLaunchOutOfResources);
    h->merge_grid_seg = h->sms * occ_fast;
    h->argmax_grid = h->sms * 2;
    h->ff_grid = h->sms * 4;
    if ((e = cudaMalloc(&h->partials, sizeof(Best) * h->argmax_grid)) != cudaSuccess) return bail("cudaMalloc partials", e);
    memset(h->h_ctl, 0, sizeof(Ctl));
    h->h_ctl->epoch = 1;
    h->h_ctl->found_pos = POS_NONE;
    if ((e = cudaMemcpy(h->ctl, h->h_ctl, sizeof(Ctl), cudaMemcpyHostToDevice)) != cudaSuccess) return bail("cudaMemcpy ctl", e);
    *out = h;
    return BPE_OK;
}

extern "C" int bpe_destroy(bpe_handle *h) {
    if (!h) return BPE_OK;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    for (int i = 0; i < 2; ++i) if (h->buf[i]) cudaFree(h->buf[i]);
    for (cudaEvent_t e : h->ev_pool) cudaEventDestroy(e);
    free_table(h, h->table);
    if (h->desc) cudaFree(h->desc);
    for (int i = 0; i < 2; ++i) if (h->edge[i]) cudaFree(h->edge[i]);
    if (h->seg_offs) cudaFree(h->seg_offs);
    if (h->sig) cudaFree(h->sig);
    if (h->cand) cudaFree(h->cand);
    if (h->delta) cudaFree(h->delta);
    if (h->dense) cudaFree(h->dense);
    if (h->dense2) cudaFree(h->dense2);
    if (h->d_cmp) cudaFree(h->d_cmp);
    if (h->d_err) cudaFree(h->d_err);
    if (h->log_pairs) cudaFree(h->log_pairs);
    if (h->log_counts) cudaFree(h->log_counts);
    if (h->partials) cudaFree(h->partials);
    if (h->d_cls) cudaFree(h->d_cls);
    if (h->d_contr) cudaFree(h->d_contr);
    if (h->d_present) cudaFree(h->d_present);
    xchg_release(h);
    enc2_free(h);
    spec_free(h);
    gen_free(h);
    if (h->enc_scratch) bpe_destroy(h->enc_scratch);
    if (h->split_slab) cudaFree(h->split_slab);
    if (h->ctl) cudaFree(h->ctl);
    if (h->h_ctl) cudaFreeHost(h->h_ctl);
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    delete h;
    return BPE_OK;
}

extern "C" int bpe_set_option(bpe_handle *h, int opt, int64_t value) {
    if (!h) return BPE_ERR_ARG;
    switch (opt) {
        case BPE_OPT_KERNEL_TIMING: h->opt_kernel_timing = value != 0; break;
        case BPE_OPT_RESCAN: h->opt_rescan = value != 0; break;
        case BPE_OPT_BATCH: h->opt_batch = (int)std::max<int64_t>(1, std::min<int64_t>(value, 4096)); break;
        case BPE_OPT_TABLE_LOG2:
            if (value != 0 && (value < 10 || value > 30)) return fail(h, BPE_ERR_ARG, "table log2 must be 0 or in [10,30]");
            h->opt_table_log2 = (int)value; break;
        case BPE_OPT_VOCAB_CAP:
            if (value < 0 || value >= 0x3fffffff) return fail(h, BPE_ERR_ARG, "vocabulary capacity out of range");
            h->opt_vocab_cap = (u32)value; break;
        case BPE_OPT_ENC_MEMO_LOG2:
            if (value != 0 && (value < 6 || value > 28)) return fail(h, BPE_ERR_ARG, "memo log2 must be 0 or in [6,28]");
            h->opt_memo_log2 = (int)value;
            cudaSetDevice(h->device); cudaStreamSynchronize(h->stream);
            enc2_free(h);   // re-created with the new size by the next encode call
            break;
        case BPE_OPT_SEG_FILTER:
            if (value < 0 || value > 2) return fail(h, BPE_ERR_ARG, "segment filter must be 0 (off), 1 (when sparse) or 2 (always)");
            h->opt_seg_filter = (int)value; h->filt_active = false; h->sig_valid = false;
            break;
        case BPE_OPT_HIST_KERNEL:
            if (value < 0 || value > 2) return fail(h, BPE_ERR_ARG, "hist kernel must be 0 (auto), 1 (packed) or 2 (hashed)");
            h->opt_hist_kernel = (int)value;
            if (value == 0) h->hist_mode = 0;
            break;
        case BPE_OPT_SPLIT_PATTERN:
            if (value != 0 && value != 1) return fail(h, BPE_ERR_ARG, "split pattern must be 0 (GPT-4) or 1 (GPT-2)");
            h->opt_split_pattern = (int)value; break;
        case BPE_OPT_SPLIT_PIECE:
            if (value != 0 && value < 4096) return fail(h, BPE_ERR_ARG, "split piece must be 0 (default) or >= 4096 bytes");
            g_split_piece_override = (u64)value; break;
        default: return fail(h, BPE_ERR_ARG, "unknown option");
    }
    return BPE_OK;
}

extern "C" int bpe_get_timing(bpe_handle *h, bpe_timing *out) {
    if (!h || !out) return BPE_ERR_ARG;
    *out = h->tm;
    return BPE_OK;
}

// ------------------------------------------------------------------------------------------------
// stream buffers
static int ensure_stream_capacity(bpe_handle *h, u64 n) {
    // round up to whole tiles (+ slack) so 16-byte loads at the tail stay inside the allocation
    const u64 need = ((n + MG_TILE - 1) / MG_TILE + 1) * MG_TILE;
    if (need > h->cap_tokens) {
        if (h->split_slab) { cudaFree(h->split_slab); h->split_slab = nullptr; h->split_cap = 0; }   // make room first
        for (int i = 0; i < 2; ++i) { if (h->buf[i]) cudaFree(h->buf[i]); h->buf[i] = nullptr; }
        h->cap_tokens = 0;
        for (int i = 0; i < 2; ++i) CU(cudaMalloc(&h->buf[i], need * 4));
        h->cap_tokens = need;
    }
    const u64 tiles = need / MG_TILE + 1;
    if (tiles > h->desc_cap) {
        if (h->desc) cudaFree(h->desc);
        h->desc = nullptr; h->desc_cap = 0;
        CU(cudaMalloc(&h->desc, tiles * 8));
        CU(cudaMemsetAsync(h->desc, 0, tiles * 8, h->stream));
        h->desc_cap = tiles;
    }
    const u64 segs = need / SEG_TOKENS + 1;
    if (segs > h->seg_cap) {
        for (int i = 0; i < 2; ++i) { if (h->edge[i]) cudaFree(h->edge[i]); h->edge[i] = nullptr; }
        if (h->seg_offs) cudaFree(h->seg_offs);
        h->seg_offs = nullptr; h->seg_cap = 0;
        for (int i = 0; i < 2; ++i) CU(cudaMalloc(&h->edge[i], segs * sizeof(Edge)));
        CU(cudaMalloc(&h->seg_offs, segs * 8));
        h->seg_cap = segs;
    }
    return BPE_OK;
}

// edge records for a stream that was just written contiguously into the current buffer
static int build_edges(bpe_handle *h, u64 n) {
    const u64 nseg = (n + SEG_TOKENS - 1) / SEG_TOKENS;
    k_build_edges<<<grid_for(nseg, 256, h->sms * 4), 256, 0, h->stream>>>(h->buf[0], h->buf[1], h->ctl, h->edge[0], 0);
    CU(cudaGetLastError());
    return BPE_OK;
}

// pack the segmented stream back into full segments (other ping-pong buffer becomes current)
static void enqueue_pack(bpe_handle *h, int force) {
    k_scan_counts<<<1, 1024, 0, h->stream>>>(h->ctl, h->edge[0], h->edge[1], h->seg_offs, force);
    k_gather<<<h->sms * 8, 256, 0, h->stream>>>(h->ctl, h->buf[0], h->buf[1], h->edge[0], h->edge[1], h->seg_offs, nullptr, force, 1);
    h->tm.kernel_launches += 2;
}
static void enqueue_edges_after_contig(bpe_handle *h) {
    k_build_edges<<<h->sms * 4, 256, 0, h->stream>>>(h->buf[0], h->buf[1], h->ctl, h->edge[0], 1);
    h->tm.kernel_launches += 1;
}

static int push_ctl(bpe_handle *h) {
    CU(cudaMemcpyAsync(h->ctl, h->h_ctl, sizeof(Ctl), cudaMemcpyHostToDevice, h->stream));
    return BPE_OK;
}
static int pull_ctl(bpe_handle *h) {
    CU(cudaMemcpyAsync(h->h_ctl, h->ctl, sizeof(Ctl), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return BPE_OK;
}

static int reset_ctl_for_stream(bpe_handle *h, u64 n) {
    int rc = pull_ctl(h);  // keep the epoch counter monotonic
    if (rc) return rc;
    const u32 epoch = h->h_ctl->epoch ? h->h_ctl->epoch : 1;
    memset(h->h_ctl, 0, sizeof(Ctl));
    h->h_ctl->epoch = epoch;
    h->h_ctl->n = n;
    h->h_ctl->found_pos = POS_NONE;
    h->h_ctl->first_idx = 256;
    return push_ctl(h);
}

static int check_offsets(bpe_handle *h, const uint64_t *offs, uint64_t k, uint64_t n) {
    if (!offs || k == 0) return BPE_OK;
    if (offs[0] != 0) return fail(h, BPE_ERR_ARG, "chunk_offsets[0] must be 0");
    for (u64 i = 1; i < k; ++i)
        if (offs[i] <= offs[i - 1] || offs[i] >= n) return fail(h, BPE_ERR_ARG, "chunk_offsets must be strictly increasing and < n");
    return BPE_OK;
}

// upload chunk offsets piecewise and mark the chunk starts in buf[0]
static int mark_chunks(bpe_handle *h, u32 *dst, const uint64_t *offs, uint64_t k, uint64_t n) {
    u64 zero = 0;
    if (!offs || k == 0) { offs = &zero; k = n ? 1 : 0; }
    if (k == 0) return BPE_OK;
    const u64 piece = 1ull << 24;  // 16M offsets = 128 MB per piece
    u64 *d_offs = nullptr;
    CU(cudaMalloc(&d_offs, std::min(piece, k) * 8));
    for (u64 s = 0; s < k; s += piece) {
        const u64 m = std::min(piece, k - s);
        cudaError_t e = cudaMemcpyAsync(d_offs, offs + s, m * 8, cudaMemcpyHostToDevice, h->stream);
        if (e == cudaSuccess) {
            k_set_flags<<<grid_for(m, 256, h->sms * 8), 256, 0, h->stream>>>(dst, d_offs, m, n);
            e = cudaStreamSynchronize(h->stream);
        }
        if (e != cudaSuccess) { cudaFree(d_offs); return fail(h, BPE_ERR_CUDA, std::string("mark_chunks: ") + cudaGetErrorString(e)); }
        h->tm.h2d_bytes += m * 8;
    }
    cudaFree(d_offs);
    return BPE_OK;
}

static int load_bytes_into(bpe_handle *h, u32 *dst, const uint8_t *bytes, uint64_t n, const unsigned char *d_perm) {
    const u64 piece = 1ull << 28;  // 256 MiB of text per staging copy
    unsigned char *d_bytes = nullptr;
    if (n == 0) return BPE_OK;
    CU(cudaMalloc(&d_bytes, std::min(piece, n)));
    for (u64 s = 0; s < n; s += piece) {
        const u64 m = std::min(piece, n - s);
        cudaError_t e = cudaMemcpyAsync(d_bytes, bytes + s, m, cudaMemcpyHostToDevice, h->stream);
        if (e == cudaSuccess) {
            k_widen_bytes<<<grid_for(m / 16 + 1, 256, h->sms * 8), 256, 0, h->stream>>>(d_bytes, dst + s, m, d_perm);
            e = cudaStreamSynchronize(h->stream);
        }
        if (e != cudaSuccess) { cudaFree(d_bytes); return fail(h, BPE_ERR_CUDA, std::string("load_bytes: ") + cudaGetErrorString(e)); }
        h->tm.h2d_bytes += m;
    }
    cudaFree(d_bytes);
    return BPE_OK;
}

extern "C" int bpe_load_stream(bpe_handle *h, const uint8_t *bytes, uint64_t n, const uint64_t *chunk_offsets,
                               uint64_t n_chunks) {
    if (!h) return BPE_ERR_ARG;
    if (!bytes && n) return fail(h, BPE_ERR_ARG, "bytes is NULL");
    if (n >= (1ull << 36)) return fail(h, BPE_ERR_ARG, "stream too long (limit 2^36 tokens)");
    CU(cudaSetDevice(h->device));
    int rc = check_offsets(h, chunk_offsets, n_chunks, n);
    if (rc) return rc;
    h->tm.h2d_bytes = 0;
    h->loaded = false; h->table_valid = false;
    if ((rc = ensure_stream_capacity(h, n))) return rc;
    if ((rc = load_bytes_into(h, h->buf[0], bytes, n, nullptr))) return rc;
    if ((rc = mark_chunks(h, h->buf[0], chunk_offsets, n_chunks, n))) return rc;
    if ((rc = reset_ctl_for_stream(h, n))) return rc;
    if ((rc = build_edges(h, n))) return rc;
    h->loaded = true; h->bytes_only = true; h->max_id = 255;
    return BPE_OK;
}

extern "C" int bpe_load_ids(bpe_handle *h, const int32_t *ids, uint64_t n, const uint64_t *chunk_offsets,
                            uint64_t n_chunks) {
    if (!h) return BPE_ERR_ARG;
    if (!ids && n) return fail(h, BPE_ERR_ARG, "ids is NULL");
    if (n >= (1ull << 36)) return fail(h, BPE_ERR_ARG, "stream too long (limit 2^36 tokens)");
    CU(cudaSetDevice(h->device));
    int rc = check_offsets(h, chunk_offsets, n_chunks, n);
    if (rc) return rc;
    h->tm.h2d_bytes = 0;
    h->loaded = false; h->table_valid = false;
    if ((rc = ensure_stream_capacity(h, n))) return rc;
    h->max_id = 0;
    if (n) {
        // stage through buf[1] (same size), then convert into buf[0]
        CU(cudaMemcpyAsync(h->buf[1], ids, n * 4, cudaMemcpyHostToDevice, h->stream));
        CU(cudaMemsetAsync(h->d_err, 0, 8, h->stream));
        k_copy_ids<<<grid_for(n, 256, h->sms * 8), 256, 0, h->stream>>>((const int *)h->buf[1], h->buf[0], n, h->d_err);
        u32 bad[2] = {0, 0};
        CU(cudaMemcpyAsync(bad, h->d_err, 8, cudaMemcpyDeviceToHost, h->stream));
        CU(cudaStreamSynchronize(h->stream));
        if (bad[0]) return fail(h, BPE_ERR_ARG, "ids must be in [0, 2^31-1)");
        h->max_id = bad[1];
        h->tm.h2d_bytes += n * 4;
    }
    if ((rc = mark_chunks(h, h->buf[0], chunk_offsets, n_chunks, n))) return rc;
    if ((rc = reset_ctl_for_stream(h, n))) return rc;
    if ((rc = build_edges(h, n))) return rc;
    h->loaded = true; h->bytes_only = false;
    return BPE_OK;
}

extern "C" int bpe_stream_len(bpe_handle *h, uint64_t *n) {
    if (!h || !n) return BPE_ERR_ARG;
    if (!h->loaded) return fail(h, BPE_ERR_STATE, "no stream loaded");
    CU(cudaSetDevice(h->device));
    int rc = pull_ctl(h);
    if (rc) return rc;
    *n = h->h_ctl->n;
    return BPE_OK;
}

extern "C" int bpe_read_stream(bpe_handle *h, int32_t *out, uint64_t cap, uint64_t *n) {
    if (!h || !n) return BPE_ERR_ARG;
    if (!h->loaded) return fail(h, BPE_ERR_STATE, "no stream loaded");
    CU(cudaSetDevice(h->device));
    int rc = pull_ctl(h);
    if (rc) return rc;
    const u64 len = h->h_ctl->n;
    *n = len;
    if (cap < len) return fail(h, BPE_ERR_CAPACITY, "output buffer too small");
    if (len == 0) return BPE_OK;
    if (!out) return fail(h, BPE_ERR_ARG, "out is NULL");
    const u32 cur = h->h_ctl->cur;
    // pack the segments into the idle ping-pong buffer (the stream itself stays as it is), strip
    // the chunk marks there, copy out
    k_scan_counts<<<1, 1024, 0, h->stream>>>(h->ctl, h->edge[0], h->edge[1], h->seg_offs, 1);
    k_gather<<<h->sms * 8, 256, 0, h->stream>>>(h->ctl, h->buf[0], h->buf[1], h->edge[0], h->edge[1], h->seg_offs,
                                                 h->buf[cur ^ 1], 1, 0);
    k_strip_flags<<<grid_for(len, 256, h->sms * 8), 256, 0, h->stream>>>(h->buf[cur ^ 1], (int *)h->buf[cur ^ 1], len);
    CU(cudaMemcpyAsync(out, h->buf[cur ^ 1], len * 4, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    h->tm.d2h_bytes = len * 4;
    return BPE_OK;
}

// ------------------------------------------------------------------------------------------------
// get_stats (base.py:13-22)
extern "C" int bpe_get_stats(bpe_handle *h, int32_t *pairs, int64_t *counts, uint64_t cap, uint64_t *n_pairs) {
    if (!h || !n_pairs) return BPE_ERR_ARG;
    if (!h->loaded) return fail(h, BPE_ERR_STATE, "no stream loaded");
    CU(cudaSetDevice(h->device));
    int rc = pull_ctl(h);
    if (rc) return rc;
    const u64 n = h->h_ctl->n;
    // distinct pairs <= n - 1; keep the load factor <= 0.5
    const u64 tcap = next_pow2(std::max<u64>(1024, 2 * n));
    Table t;
    if ((rc = alloc_table(h, t, tcap, true))) { free_table(h, t); return rc; }
    const u64 used_before = h->h_ctl->table_used;
    {   // the scratch table counts its own occupancy (k_hist_hash refuses inserts near a full table)
        const ull zero = 0;
        CU(cudaMemcpyAsync(&h->ctl->table_used, &zero, 8, cudaMemcpyHostToDevice, h->stream));
    }
    k_hist_hash<<<h->sms * 8, 256, 0, h->stream>>>(h->buf[0], h->buf[1], h->ctl, h->edge[0], h->edge[1], t, 0);
    std::vector<u64> keys(tcap), cnt(tcap), first(tcap);
    cudaError_t e = cudaMemcpyAsync(keys.data(), t.keys, tcap * 8, cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(cnt.data(), t.counts, tcap * 8, cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(first.data(), t.first, tcap * 8, cudaMemcpyDeviceToHost, h->stream);
    // k_hist_hash bumped ctl->table_used for the scratch table: restore it
    h->h_ctl->table_used = used_before;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&h->ctl->table_used, &h->h_ctl->table_used, 8, cudaMemcpyHostToDevice, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    free_table(h, t);
    if (e != cudaSuccess) return fail(h, BPE_ERR_CUDA, std::string("bpe_get_stats: ") + cudaGetErrorString(e));
    std::vector<u64> order;
    for (u64 i = 0; i < tcap; ++i) if (keys[i] != KEY_EMPTY) order.push_back(i);
    std::sort(order.begin(), order.end(), [&](u64 x, u64 y) { return first[x] < first[y]; });
    *n_pairs = order.size();
    h->tm.d2h_bytes = tcap * 24;
    if (order.size() > cap) return fail(h, BPE_ERR_CAPACITY, "pairs/counts buffers too small");
    for (u64 i = 0; i < order.size(); ++i) {
        pairs[2 * i] = (int32_t)(keys[order[i]] >> 32);
        pairs[2 * i + 1] = (int32_t)(keys[order[i]] & 0xffffffffu);
        counts[i] = (int64_t)cnt[order[i]];
    }
    return BPE_OK;
}

// ------------------------------------------------------------------------------------------------
// merge (base.py:25-41), single step
// One merge over the stream.  Pairs a != b: the segmented in-place pass.  Pairs (a,a) need the
// run-parity carry along the stream, so they pack the stream and use the contiguous kernel
// (which also refills every segment).  Every kernel gates itself on the device-resident pair, so
// the whole sequence is enqueued unconditionally; `same` >= 0 lets the host skip the no-ops when
// it knows the pair (single-step API).
static void launch_merge(bpe_handle *h, ull *delta, int force, int same = -1, bool use_xchg = false) {
    const unsigned char *xbase = use_xchg ? h->xchg : nullptr;
    if (same != 1) {
        SegArgs S;
        S.ctl = h->ctl; S.buf0 = h->buf[0]; S.buf1 = h->buf[1]; S.e0 = h->edge[0]; S.e1 = h->edge[1];
        S.delta = delta; S.V = h->V; S.force = force; S.xbase = xbase; S.xstride = h->xchg_stride;
        if (h->filt_active) k_merge_seg<true><<<h->merge_grid_seg, MS_THREADS, MS_SMEM_BYTES, h->stream>>>(S);
        else k_merge_seg<false><<<h->merge_grid_seg, MS_THREADS, MS_SMEM_BYTES, h->stream>>>(S);
        h->tm.kernel_launches += 1;
    }
    if (same != 0) {
        MergeArgs A;
        A.ctl = h->ctl; A.buf0 = h->buf[0]; A.buf1 = h->buf[1]; A.desc = h->desc; A.delta = delta; A.V = h->V; A.force = force;
        A.xbase = xbase; A.xstride = h->xchg_stride;
        enqueue_pack(h, force);
        k_merge<true><<<h->merge_grid_same, MG_THREADS, 0, h->stream>>>(A);
        h->tm.kernel_launches += 1;
        enqueue_edges_after_contig(h);
        if (h->filt_active) {      // the pack moved tokens between segments: signatures from the tokens again (gated on a == b)
            k_sig_build<<<h->sms * 8, 256, 0, h->stream>>>(h->buf[0], h->buf[1], h->ctl, h->edge[0], h->edge[1], h->sig, 1);
            h->tm.kernel_launches += 1;
        }
    }
}

extern "C" int bpe_merge(bpe_handle *h, int32_t a, int32_t b, int32_t idx, uint64_t *new_len) {
    if (!h) return BPE_ERR_ARG;
    if (!h->loaded) return fail(h, BPE_ERR_STATE, "no stream loaded");
    if (a < 0 || b < 0 || idx < 0 || a == 0x7fffffff || b == 0x7fffffff || idx == 0x7fffffff)
        return fail(h, BPE_ERR_ARG, "ids must be in [0, 2^31-1)");
    CU(cudaSetDevice(h->device));
    int rc = pull_ctl(h);
    if (rc) return rc;
    h->h_ctl->a = a; h->h_ctl->b = b; h->h_ctl->z = idx;
    if ((rc = push_ctl(h))) return rc;
    launch_merge(h, nullptr, 1, a == b ? 1 : 0);
    CU(cudaGetLastError());
    if ((rc = pull_ctl(h))) return rc;
    h->table_valid = false;
    if (idx > 255) h->bytes_only = false;
    h->max_id = std::max(h->max_id, (u32)idx);
    if (new_len) *new_len = h->h_ctl->n;
    return BPE_OK;
}

// ------------------------------------------------------------------------------------------------
// training loop (basic.py:31-45 / regex.py:49-66)
// The table starts small (the arg-max scans every slot each iteration) and doubles on demand:
// k_apply_delta stops inserting at ctl->table_limit and raises ctl->overflow (handle_overflow).
static u64 auto_table_cap(bpe_handle *h, u64 n_unbounded_inserts) {
    if (h->opt_table_log2) return 1ull << h->opt_table_log2;
    u64 c = 1ull << 17;   // a byte stream has at most 65536 distinct pairs
    while (c < 2 * n_unbounded_inserts + 2) c <<= 1;
    return c;
}
#define TABLE_MAX_LOAD 0.6

// The owned delta vector must cover vocabulary capacity V; h->V (the layout every kernel indexes with) is
// set to exactly V.  The capacity of the owned buffer is tracked separately: the step API points the
// kernels at a caller's buffer and changes h->V without touching h->delta.
static int ensure_delta(bpe_handle *h, u32 V) {
    if (!h->delta || h->delta_cap < V) {
        if (h->delta) cudaFree(h->delta);
        h->delta = nullptr; h->delta_cap = 0;
        CU(cudaMalloc(&h->delta, (2ull * V + 1) * 8));
        h->delta_cap = V;
    }
    if (h->V != V) CU(cudaMemsetAsync(h->delta, 0, (2ull * h->delta_cap + 1) * 8, h->stream));   // layout changes: all zero again
    h->V = V;
    return BPE_OK;
}

// Byte-pair histogram of the current (byte) stream into dense_out[65536] (zeroed by the caller).
// k_hist_dense_packed (dense 16-bit counters in 128 KB of shared memory) replaces k_hist_dense (hashed per-block table +
// __match_any_sync folding, 19 ms per GiB).  It was written when no GPU was reachable and has only run on the CPU SIMT
// emulator, so a handle's first histogram of a LARGE stream (>= 8 Mi tokens; smaller ones just take k_hist_dense) runs both
// kernels, timed with events, and compares all 65,536 counters on the device: equal and not slower -> the packed kernel
// from then on; otherwise (or 128 KB of shared memory refused) -> k_hist_dense stays.  bpe_timing.hist_kernel
// reports which one is in use.  (Drop the cross-check once `pytest -m gpu` has passed on a B200 with hist_kernel == 1.)
#define HIST_DECIDE_MIN_TOKENS (8ull << 20)   /* smaller streams say nothing about speed: they take k_hist_dense, undecided */
static int hist_dense(bpe_handle *h, ull *dense_out) {
    const int grid_old = h->sms * 3;
    if (h->opt_hist_kernel && h->hist_mode != h->opt_hist_kernel) {      // BPE_OPT_HIST_KERNEL: forced (tests)
        if (h->opt_hist_kernel == 1 &&
            cudaFuncSetAttribute(k_hist_dense_packed, cudaFuncAttributeMaxDynamicSharedMemorySize, HP_SMEM_BYTES) != cudaSuccess)
            return fail(h, BPE_ERR_CUDA, "k_hist_dense_packed: 128 KB of shared memory refused");
        h->hist_mode = h->opt_hist_kernel;
    }
    if (h->hist_mode == 0 && h->h_ctl->n >= HIST_DECIDE_MIN_TOKENS) {
        h->hist_mode = 2;
        if (cudaFuncSetAttribute(k_hist_dense_packed, cudaFuncAttributeMaxDynamicSharedMemorySize, HP_SMEM_BYTES) == cudaSuccess) {
            if (!h->dense2) CU(cudaMalloc(&h->dense2, 65536 * 8));
            if (!h->d_cmp) CU(cudaMalloc(&h->d_cmp, 4));
            CU(cudaMemsetAsync(h->dense2, 0, 65536 * 8, h->stream));
            CU(cudaMemsetAsync(h->d_cmp, 0, 4, h->stream));
            cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
            for (auto &e : ev) CU(cudaEventCreate(&e));
            auto drop_events = [&]() { for (auto &e : ev) cudaEventDestroy(e); };
            cudaEventRecord(ev[0], h->stream);
            k_hist_dense<<<grid_old, 256, 0, h->stream>>>(h->buf[0], h->buf[1], h->ctl, h->edge[0], h->edge[1], dense_out, h->d_err);
            cudaEventRecord(ev[1], h->stream);
            if (cudaGetLastError() != cudaSuccess) { drop_events(); return fail(h, BPE_ERR_CUDA, "k_hist_dense launch failed"); }
            k_hist_dense_packed<<<h->sms, HP_THREADS, HP_SMEM_BYTES, h->stream>>>(h->buf[0], h->buf[1], h->ctl, h->edge[0], h->edge[1], h->dense2, h->d_err);
            cudaEventRecord(ev[2], h->stream);
            if (cudaGetLastError() != cudaSuccess) {      // the launch itself was refused (a launch error is not sticky): keep k_hist_dense
                drop_events();
                h->tm.kernel_launches += 1;
                h->tm.hist_kernel = 2;
                return BPE_OK;
            }
            k_dense_compare<<<65536 / 256, 256, 0, h->stream>>>(dense_out, h->dense2, h->d_cmp);
            h->tm.kernel_launches += 3;
            u32 differ = 1;
            cudaError_t e = cudaMemcpyAsync(&differ, h->d_cmp, 4, cudaMemcpyDeviceToHost, h->stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
            float ms_old = 0, ms_new = 0;
            if (e == cudaSuccess) { cudaEventElapsedTime(&ms_old, ev[0], ev[1]); cudaEventElapsedTime(&ms_new, ev[1], ev[2]); }
            drop_events();
            if (e != cudaSuccess) return fail(h, BPE_ERR_CUDA, std::string("hist_dense: ") + cudaGetErrorString(e));
            // adopted only when it gives the same 65,536 counters AND is not slower on this very stream
            if (!differ && ms_new <= ms_old) h->hist_mode = 1;
            h->tm.hist_kernel = (uint64_t)h->hist_mode;
            return BPE_OK;      // dense_out holds k_hist_dense's result either way
        }
    }
    if (h->hist_mode == 1)
        k_hist_dense_packed<<<h->sms, HP_THREADS, HP_SMEM_BYTES, h->stream>>>(h->buf[0], h->buf[1], h->ctl, h->edge[0], h->edge[1], dense_out, h->d_err);
    else
        k_hist_dense<<<grid_old, 256, 0, h->stream>>>(h->buf[0], h->buf[1], h->ctl, h->edge[0], h->edge[1], dense_out, h->d_err);
    h->tm.kernel_launches += 1;
    h->tm.hist_kernel = (uint64_t)h->hist_mode;
    return BPE_OK;
}

// (re)build the pair-count table from the current stream
static int build_table(bpe_handle *h, u64 cap) {
    int rc;
    if (!h->table.keys || h->table.mask + 1 != cap) {
        free_table(h, h->table);
        if ((rc = alloc_table(h, h->table, cap, false))) return rc;
    } else {
        CU(cudaMemsetAsync(h->table.keys, 0xff, cap * 8, h->stream));
        CU(cudaMemsetAsync(h->table.counts, 0, cap * 8, h->stream));
    }
    const ull zero = 0;
    CU(cudaMemcpyAsync(&h->ctl->table_used, &zero, 8, cudaMemcpyHostToDevice, h->stream));
    if (h->bytes_only) {
        CU(cudaMemsetAsync(h->dense, 0, 65536 * 8, h->stream));
        CU(cudaMemsetAsync(h->d_err, 0, 4, h->stream));
        if ((rc = hist_dense(h, h->dense))) return rc;
        k_dense_to_table<<<65536 / 256, 256, 0, h->stream>>>(h->dense, h->table, h->ctl);
        h->tm.kernel_launches += 1;
    } else {
        k_hist_hash<<<h->sms * 8, 256, 0, h->stream>>>(h->buf[0], h->buf[1], h->ctl, h->edge[0], h->edge[1], h->table, 0);
        h->tm.kernel_launches += 1;
    }
    CU(cudaGetLastError());
    return BPE_OK;
}

// grow / clean the table: live entries are re-inserted into a fresh table of `cap` slots
static int rehash_table(bpe_handle *h, u64 cap) {
    Table nt;
    int rc = alloc_table(h, nt, cap, false);
    if (rc) { free_table(h, nt); return rc; }
    const ull zero = 0;
    CU(cudaMemcpyAsync(&h->ctl->table_used, &zero, 8, cudaMemcpyHostToDevice, h->stream));
    k_rehash<<<grid_for(h->table.mask + 1, 256, h->sms * 8), 256, 0, h->stream>>>(h->table, nt, h->ctl);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(h->stream));
    free_table(h, h->table);
    h->table = nt;
    h->tm.kernel_launches++;
    return BPE_OK;
}

// fold the event pairs recorded since the last call into tm.merge_kernel_ms (stream must be idle)
static void drain_kernel_events(bpe_handle *h) {
    for (int i = 0; i + 1 < h->ev_used; i += 2) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, h->ev_pool[i], h->ev_pool[i + 1]) == cudaSuccess) h->tm.merge_kernel_ms += ms;
    }
    h->ev_used = 0;
}

static void timed_merge(bpe_handle *h, ull *delta, bool use_xchg = false) {
    if (!h->opt_kernel_timing) { launch_merge(h, delta, 0, -1, use_xchg); return; }
    while ((int)h->ev_pool.size() < h->ev_used + 2) { cudaEvent_t e; cudaEventCreate(&e); h->ev_pool.push_back(e); }
    cudaEventRecord(h->ev_pool[h->ev_used], h->stream);
    launch_merge(h, delta, 0, -1, use_xchg);
    cudaEventRecord(h->ev_pool[h->ev_used + 1], h->stream);
    h->ev_used += 2;
}

// ctl->overflow was raised by k_apply_delta: some delta entries of the last performed merge are
// still pending.  Double the table (dead pairs are dropped on the way), re-run the apply.
static int handle_overflow(bpe_handle *h) {
    int rc;
    while (h->h_ctl->overflow) {
        const u64 new_cap = (h->table.mask + 1) * 2;
        if ((rc = rehash_table(h, new_cap))) return rc;
        if ((rc = pull_ctl(h))) return rc;
        h->h_ctl->overflow = 0;
        h->h_ctl->table_limit = (u64)(TABLE_MAX_LOAD * (double)new_cap);
        if ((rc = push_ctl(h))) return rc;
        k_apply_delta<<<(h->V + 255) / 256, 256, 0, h->stream>>>(h->table, h->ctl, h->delta, h->V, 0, 0, 0, 1, 1);
        h->tm.kernel_launches++;
        if ((rc = pull_ctl(h))) return rc;
    }
    return BPE_OK;
}

// Between batches: when merges have emptied the segments below half full on average, pack the
// stream into full segments again (fewer, fuller segments = less per-segment overhead).
static void maybe_repack(bpe_handle *h) {
    const u64 nseg = h->h_ctl->nseg;
    if (nseg < 64 || h->h_ctl->contig) return;
    if (2 * h->h_ctl->n >= nseg * (u64)SEG_TOKENS) return;
    enqueue_pack(h, 1);
    enqueue_edges_after_contig(h);
    if (h->filt_active) {
        k_sig_build<<<h->sms * 8, 256, 0, h->stream>>>(h->buf[0], h->buf[1], h->ctl, h->edge[0], h->edge[1], h->sig, 0);
        h->tm.kernel_launches += 1;
    }
}

// ---- segment filter (k_seg_filter.cuh) ---------------------------------------------------------------------------
static void filt_rebuild(bpe_handle *h, int gate_same) {
    k_sig_build<<<h->sms * 8, 256, 0, h->stream>>>(h->buf[0], h->buf[1], h->ctl, h->edge[0], h->edge[1], h->sig, gate_same);
    h->tm.kernel_launches += 1;
}

// switch the filter on for the iterations enqueued from here on: storage, list address in the control block, signatures
// of the stream as it is now
static int filt_activate(bpe_handle *h) {
    const u64 want = (u64)h->h_ctl->nseg + 64;      // segments of the stream as it is now (the count only ever falls), not the buffers' capacity
    if (h->sig_cap < want) {
        if (h->sig) cudaFree(h->sig);
        if (h->cand) cudaFree(h->cand);
        h->sig = nullptr; h->cand = nullptr; h->sig_cap = 0;
        CU(cudaMalloc(&h->sig, want * SIG_WORDS * 4));
        CU(cudaMalloc(&h->cand, want * 4));
        h->sig_cap = want;
    }
    const u64 ptr = (u64)(uintptr_t)h->cand;
    const u32 zero = 0;
    CU(cudaMemcpyAsync(&h->ctl->cand_ptr, &ptr, 8, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(&h->ctl->n_cand, &zero, 4, cudaMemcpyHostToDevice, h->stream));
    CU(cudaStreamSynchronize(h->stream));          // `ptr` / `zero` are stack variables
    h->h_ctl->cand_ptr = ptr; h->h_ctl->n_cand = 0;
    filt_rebuild(h, 0);
    h->filt_active = true;
    return BPE_OK;
}

static void enqueue_iteration(bpe_handle *h) {
    if (h->opt_rescan) {
        // verification mode: rebuild the histogram from the stream, no incremental update
        cudaMemsetAsync(h->table.keys, 0xff, (h->table.mask + 1) * 8, h->stream);
        cudaMemsetAsync(h->table.counts, 0, (h->table.mask + 1) * 8, h->stream);
        cudaMemsetAsync(&h->ctl->table_used, 0, 8, h->stream);
        k_hist_hash<<<h->sms * 4, 256, 0, h->stream>>>(h->buf[0], h->buf[1], h->ctl, h->edge[0], h->edge[1], h->table, 1);
        h->tm.kernel_launches++;
    }
    if (h->filt_active) { k_cand_reset<<<1, 1, 0, h->stream>>>(h->ctl); h->tm.kernel_launches++; }
    k_argmax<<<h->argmax_grid, 256, 0, h->stream>>>(h->table, h->ctl, h->partials, h->log_pairs, h->log_counts);
    k_find_first<<<h->ff_grid, 256, 0, h->stream>>>(h->buf[0], h->buf[1], h->edge[0], h->edge[1], h->table, h->ctl, h->log_pairs, h->log_counts, 0);
    h->tm.kernel_launches += 2;
    if (h->filt_active) {    // candidate segments of the selected pair; k_merge_seg<true> works through that list only
        k_seg_filter<<<h->sms * 8, 256, 0, h->stream>>>(h->ctl, h->edge[0], h->edge[1], h->edge[0], h->edge[1], h->sig, h->cand);
        h->tm.kernel_launches++;
    }
    if (h->opt_rescan) timed_merge(h, nullptr);
    else {
        timed_merge(h, h->delta);
        k_apply_delta<<<(h->V + 255) / 256, 256, 0, h->stream>>>(h->table, h->ctl, h->delta, h->V, 0, 0, 0, 1, 0);
        h->tm.kernel_launches++;
    }
    if (h->filt_active) {    // the listed segments may have changed: their signatures from their tokens again
        k_sig_rebuild_cand<<<h->sms * 4, 256, 0, h->stream>>>(h->ctl, h->buf[0], h->buf[1], h->edge[0], h->edge[1], h->sig, h->cand);
        h->tm.kernel_launches++;
    }
}

extern "C" int bpe_train(bpe_handle *h, int32_t num_merges, int32_t first_idx, int32_t *out_pairs, int64_t *out_counts,
                         int32_t *n_done) {
    if (!h || !n_done) return BPE_ERR_ARG;
    if (!h->loaded) return fail(h, BPE_ERR_STATE, "no stream loaded");
    if (num_merges < 0 || first_idx < 0) return fail(h, BPE_ERR_ARG, "num_merges and first_idx must be >= 0");
    if ((u64)first_idx + (u64)num_merges >= 0x7fffffffull) return fail(h, BPE_ERR_ARG, "vocabulary would exceed 2^31-1");
    if (num_merges && (!out_pairs || !out_counts)) return fail(h, BPE_ERR_ARG, "output buffers are NULL");
    CU(cudaSetDevice(h->device));
    *n_done = 0;
    h->tm.kernel_launches = 0; h->tm.d2h_bytes = 0; h->tm.merge_kernel_ms = 0;
    if (num_merges == 0) return BPE_OK;
    int rc = pull_ctl(h);
    if (rc) return rc;
    // the delta vector is indexed by the ids of a merge's neighbours: it must cover every id of the loaded
    // stream (bpe_load_ids accepts any id < 2^31-1) as well as the ids this call creates
    if ((u64)h->max_id + 1 >= 0x7fffffffull / 2) return fail(h, BPE_ERR_ARG, "bpe_train: ids of the loaded stream are too large for the dense delta vector");
    const u32 V = std::max(std::max((u32)first_idx + (u32)num_merges, h->max_id + 1), h->opt_vocab_cap);
    if ((rc = ensure_delta(h, V))) return rc;
    if (h->log_cap < num_merges) {
        if (h->log_pairs) cudaFree(h->log_pairs);
        if (h->log_counts) cudaFree(h->log_counts);
        h->log_pairs = nullptr; h->log_counts = nullptr; h->log_cap = 0;
        CU(cudaMalloc(&h->log_pairs, (size_t)num_merges * 8));
        CU(cudaMalloc(&h->log_counts, (size_t)num_merges * 8));
        h->log_cap = num_merges;
    }
    cudaEvent_t ev0, ev1, ev2;
    CU(cudaEventCreate(&ev0)); CU(cudaEventCreate(&ev1)); CU(cudaEventCreate(&ev2));

    // ---- initial statistics (the only full histogram of the run) ----
    CU(cudaEventRecord(ev0, h->stream));
    // only a non-byte stream (bpe_load_ids) or the rescan mode insert without the load check
    u64 cap = auto_table_cap(h, !h->bytes_only ? h->h_ctl->n : 0);
    if (h->opt_rescan && !h->opt_table_log2) {   // every iteration clears and rescans: keep the table moderate
        cap = 1ull << 20;
        while (cap < h->h_ctl->n / 16 && cap < (1ull << 26)) cap <<= 1;
    }
    const bool reuse = h->table_valid && h->table.keys && !h->opt_rescan;  // continuing a previous bpe_train
    if (!reuse && (rc = build_table(h, cap))) return rc;
    h->table_valid = false;  // becomes true again when the loop ends cleanly
    u32 bad = 0;
    if (!reuse && h->bytes_only) CU(cudaMemcpyAsync(&bad, h->d_err, 4, cudaMemcpyDeviceToHost, h->stream));
    if ((rc = pull_ctl(h))) return rc;  // refreshes table_used
    if (bad) return fail(h, BPE_ERR_INTERNAL, "byte stream contains ids >= 256");
    h->h_ctl->iter = 0; h->h_ctl->done = 0; h->h_ctl->first_idx = (u32)first_idx; h->h_ctl->max_iter = (u32)num_merges;
    h->h_ctl->sum_in = 0; h->h_ctl->sum_out = 0;
    h->h_ctl->cand_sum = 0; h->h_ctl->seg_sum = 0;
    h->h_ctl->overflow = 0;
    h->h_ctl->table_limit = (u64)(TABLE_MAX_LOAD * (double)(h->table.mask + 1));
    if ((rc = push_ctl(h))) return rc;
    CU(cudaEventRecord(ev1, h->stream));

    // ---- the merge loop: batches of iterations enqueued back to back, one host sync per batch ----
    int done_iters = 0;
    bool exhausted = false;
    h->filt_active = false;
    if (h->opt_seg_filter == 2 && !h->opt_rescan && (rc = filt_activate(h))) return rc;
    u64 drops_seen = 0;
    while (done_iters < num_merges && !exhausted) {
        const int k = std::min(h->opt_batch, num_merges - done_iters);
        maybe_repack(h);
        for (int i = 0; i < k; ++i) enqueue_iteration(h);
        CU(cudaGetLastError());
        if ((rc = pull_ctl(h))) return rc;
        drain_kernel_events(h);
        if (h->opt_seg_filter == 1 && !h->filt_active && !h->opt_rescan && (int)h->h_ctl->iter > done_iters) {
            // BPE_OPT_SEG_FILTER = 1: once a merge replaces, on average, fewer tokens than a thirty-second of the segments
            // there are, most segments cannot be touched by it: filter from the next batch on (merges only get sparser)
            const u64 drops = h->h_ctl->sum_in - h->h_ctl->sum_out;
            const u64 per_merge = (drops - drops_seen) / (u64)((int)h->h_ctl->iter - done_iters);
            drops_seen = drops;
            if (per_merge * 32 < h->h_ctl->nseg && (rc = filt_activate(h))) return rc;
        }
        if (h->h_ctl->overflow) {
            if (h->opt_rescan) return fail(h, BPE_ERR_CAPACITY, "rescan mode: pair table too small (set BPE_OPT_TABLE_LOG2)");
            if ((rc = handle_overflow(h))) return rc;
        }
        done_iters = (int)h->h_ctl->iter;
        exhausted = h->h_ctl->done != 0;
    }
    CU(cudaEventRecord(ev2, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    float ms01 = 0, ms12 = 0;
    cudaEventElapsedTime(&ms01, ev0, ev1);
    cudaEventElapsedTime(&ms12, ev1, ev2);
    cudaEventDestroy(ev0); cudaEventDestroy(ev1); cudaEventDestroy(ev2);
    h->tm.init_ms = ms01; h->tm.loop_ms = ms12;
    h->tm.tokens_in = h->h_ctl->sum_in; h->tm.tokens_out = h->h_ctl->sum_out;
    h->tm.table_slots = h->table.mask + 1; h->tm.table_used = h->h_ctl->table_used;
    h->tm.filter_candidates = h->h_ctl->cand_sum; h->tm.filter_segments = h->h_ctl->seg_sum;
    if (done_iters > 0) {
        CU(cudaMemcpyAsync(out_pairs, h->log_pairs, (size_t)done_iters * 8, cudaMemcpyDeviceToHost, h->stream));
        CU(cudaMemcpyAsync(out_counts, h->log_counts, (size_t)done_iters * 8, cudaMemcpyDeviceToHost, h->stream));
        CU(cudaStreamSynchronize(h->stream));
        h->tm.d2h_bytes = (u64)done_iters * 16;
    }
    *n_done = done_iters;
    h->filt_active = false;      // the other users of launch_merge (bpe_merge, replay, the step API) do not maintain signatures
    h->table_valid = !h->opt_rescan;
    if (first_idx + done_iters > 256) h->bytes_only = false;
    if (done_iters > 0) h->max_id = std::max(h->max_id, (u32)(first_idx + done_iters - 1));
    return BPE_OK;
}

// debug/test hook: dump the live entries (count > 0) of the incremental table, unordered
extern "C" int bpe_debug_table(bpe_handle *h, int32_t *pairs, int64_t *counts, uint64_t cap, uint64_t *n_pairs) {
    if (!h || !n_pairs) return BPE_ERR_ARG;
    if (!h->table.keys) return fail(h, BPE_ERR_STATE, "no table");
    CU(cudaSetDevice(h->device));
    const u64 tcap = h->table.mask + 1;
    std::vector<u64> keys(tcap), cnt(tcap);
    CU(cudaMemcpyAsync(keys.data(), h->table.keys, tcap * 8, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(cnt.data(), h->table.counts, tcap * 8, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    u64 m = 0;
    for (u64 i = 0; i < tcap; ++i) {
        if (keys[i] == KEY_EMPTY || cnt[i] == 0) continue;
        if (m < cap) { pairs[2 * m] = (int32_t)(keys[i] >> 32); pairs[2 * m + 1] = (int32_t)(keys[i] & 0xffffffffu); counts[m] = (int64_t)cnt[i]; }
        ++m;
    }
    *n_pairs = m;
    return m > cap ? fail(h, BPE_ERR_CAPACITY, "buffers too small") : BPE_OK;
}

#include "encode_host.inl"
#include "step_host.inl"
#include "special_host.inl"
#include "split_host.inl"
#include "encode2_host.inl"
#include "batch_host.inl"
#include "decode_host.inl"
