/*
 * b2f_api.cu -- C ABI (include/b2f.h) of libb200forest.so: model lifetime, the pinned-ring /
 * multi-stream staging around the kernels, timing helpers and the NCCL plumbing.
 *
 * The reference's counterpart of this file is Python glue: `lifespan` loading the model
 * (reference app/main.py:20-31), `CustomModel.load_context` / `.predict`
 * (databricks/src/02-register-model.ipynb:317-353).  Here the model is a flattened forest in HBM
 * and "predict" is H2D copy -> one fused kernel -> D2H copy, pipelined over CUDA streams.
 * There is no CPU fallback anywhere in this file: no device, no result.
 */
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>
#include <stdarg.h>
#include <stddef.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <deque>
#include <mutex>
#include <string>
#include <thread>
#include <new>
#include <unordered_map>
#include <vector>

#include "../../include/b2f.h"
#include "feature_moments.cuh"
#include "forest_blob.h"
#include "forest_predict.cuh"
#include "forest_predict_tile.cuh"
#include "forest_predict_rank.cuh"
#include "forest_rank.h"
#include "json_rows.h"
#include "row_encoder.h"

#define B2F_VERSION_STR "b200forest 0.1.0 (sm_100a)"
#define B2F_STREAMS 4
#define B2F_TICKETS 256
#define B2F_CHUNK_ROWS 16384
#define B2F_FLUSH_BYTES (256ull << 20) /* > 126 MB L2 */

/* ------------------------------------------------------------------ errors */
static thread_local char g_err[512] = "";

static int set_err(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
#define CUDA_TRY(expr)                                                                         \
    do {                                                                                       \
        cudaError_t e_ = (expr);                                                               \
        if (e_ != cudaSuccess)                                                                 \
            return set_err(B2F_ECUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

extern "C" const char *b2f_last_error(void) { return g_err; }
extern "C" const char *b2f_version(void) { return B2F_VERSION_STR; }

extern "C" int b2f_device_count(void) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) return set_err(B2F_ENODEV, "no CUDA device: %s", cudaGetErrorString(e));
    return n;
}

/* ------------------------------------------------------------------ NCCL (lazy dlopen) */
struct NcclApi {
    void *handle = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommInitAll)(ncclComm_t *, int, const int *) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)(void) = nullptr;
    ncclResult_t (*GroupEnd)(void) = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
};
static NcclApi g_nccl;

static int nccl_load(void) {
    if (g_nccl.handle) return B2F_OK;
    const char *names[] = {"libnccl.so.2", "libnccl.so"};
    void *h = nullptr;
    for (const char *nm : names) {
        h = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
        if (h) break;
    }
    if (!h) return set_err(B2F_ENCCL, "cannot dlopen libnccl.so.2: %s", dlerror());
#define LOADSYM(field, sym)                                                        \
    do {                                                                           \
        *(void **)(&g_nccl.field) = dlsym(h, sym);                                 \
        if (!g_nccl.field) return set_err(B2F_ENCCL, "NCCL symbol %s missing", sym); \
    } while (0)
    LOADSYM(GetUniqueId, "ncclGetUniqueId");
    LOADSYM(CommInitRank, "ncclCommInitRank");
    LOADSYM(CommInitAll, "ncclCommInitAll");
    LOADSYM(CommDestroy, "ncclCommDestroy");
    LOADSYM(AllGather, "ncclAllGather");
    LOADSYM(GroupStart, "ncclGroupStart");
    LOADSYM(GroupEnd, "ncclGroupEnd");
    LOADSYM(GetErrorString, "ncclGetErrorString");
#undef LOADSYM
    g_nccl.handle = h;
    return B2F_OK;
}
#define NCCL_TRY(expr)                                                                                      \
    do {                                                                                                    \
        ncclResult_t r_ = (expr);                                                                           \
        if (r_ != ncclSuccess) return set_err(B2F_ENCCL, "%s failed: %s", #expr, g_nccl.GetErrorString(r_)); \
    } while (0)

/* ------------------------------------------------------------------ model */
struct Slot {
    cudaStream_t stream = nullptr;
    void *d_rows = nullptr;
    void *d_proba = nullptr; /* 24 B per row: double, {float, int32} pairs or b2f_scored_full records */
    int32_t *d_label = nullptr;
    int64_t cap_rows = 0;
};

struct TicketRec {
    uint64_t id = 0;
    cudaEvent_t ev[B2F_STREAMS] = {nullptr, nullptr, nullptr, nullptr};
    uint32_t used_mask = 0;
};

struct b2f_model {
    int device = 0;
    int sm_count = 0;
    int max_smem_optin = 0;
    KParams kp;
    b2f_blob_header hdr;
    int walk_mode = B2F_WALK_GLOBAL;
    int smem_bytes = 0;
    int rows_per_warp_max = 2;
    int64_t chunk_rows = B2F_CHUNK_ROWS;
    std::vector<int64_t> chunk_plan; /* per-chunk share of a batch in 1/1024ths */
    /* tile kernel (large batches) */
    bool tile_ok = false;
    TParams tp;
    void *d_tile_layout = nullptr;
    TPiece *d_tile_pieces = nullptr;
    int tile_smem_bytes = 0;
    int tile_cwarps = B2F_TILE_WARPS_MIN;
    int64_t tile_min_rows = 32768;
    int64_t tile_layout_bytes = 0;
    int64_t launches_tile = 0;
    int64_t launches_split = 0;
    int64_t split_max_rows = 0;
    bool packed_ok = false;
    /* rank kernel (B2F_ROWS_RANKED rows; forest resident in its 4-byte-node complete-tree layout) */
    b2f_ranker rk;
    bool rank_ok = false;
    RParams rp;
    void *d_rank_layout = nullptr;
    int rank_smem_bytes = 0;
    int rank_u = 4;
    bool rank_stream = false; /* the rank layout streams through shared memory in pieces (too large to stay resident) */
    int64_t launches_rank = 0;
    bool rank_last_pdl = false; /* the last rank launch went out with programmatic stream serialization */
#ifdef B2F_RANK_TRACE
    unsigned long long *d_rank_trace = nullptr; /* B2F_RANK_TRACE_LAUNCHES launches x sm_count CTAs x B2F_RANK_TRACE_WORDS */
#endif
    void *d_blob = nullptr;
    int64_t forest_bytes = 0;
    b2f_model *outlier = nullptr; /* attached isolation forest (b2f_model_attach_outlier_forest): a child handle on the
                                     same device whose kernels are launched on this handle's streams and rows */
    Slot slots[B2F_STREAMS];
    cudaStream_t compute = nullptr; /* device-resident interface + moments */
    TicketRec tickets[B2F_TICKETS];
    uint64_t next_ticket = 1;
    uint64_t next_slot = 0;
    /* moments */
    void *d_mom_rows = nullptr;
    int64_t mom_cap_rows = 0;
    double *d_mom_partials = nullptr;
    int mom_blocks = 0;
    unsigned int *d_mom_ticket = nullptr;
    double *d_mom_out = nullptr;
    double *d_gather = nullptr; /* nranks * 72 doubles */
    int gather_cap = 0;
    /* L2 flush scratch */
    void *d_flush = nullptr;
    /* nccl */
    ncclComm_t comm = nullptr;
    int nranks = 0;
    int rank = 0;
    int64_t launches = 0;
};

/* the rank kernel goes out with programmatic stream serialization: back-to-back launches on one stream overlap the next
 * launch's prologue (forest fill, row staging) with this launch's tail.  The kernel waits (griddepcontrol.wait) only before its
 * first global store, so it reads its rows while earlier launches may still run -- not only the previous one: every rank launch
 * triggers its dependents at entry, so a chain of launches with the attribute can be resident at once (small grids leave SMs
 * free).  A launch whose rows overlap what any launch of the current chain writes therefore goes out without the attribute;
 * it starts only after its predecessor has completed, which completed only after its own wait, i.e. after everything before
 * it: such a launch starts a new chain.
 * How far back a chain must be remembered: a CTA passes its wait only after the previous launch has completed, and every CTA
 * passes it before it exits, so while launch A is incomplete every later launch of the chain holds a resident CTA (all of its
 * CTAs have started: the launch after it has).  At most 2 rank CTAs (1024 threads each) fit an SM, so when a new launch starts,
 * a launch more than 2 * sm_count + 1 launches back has completed and a later launch has waited for it (its writes are
 * flushed): the record keeps the chain's last 2 * sm_count + 1 launches and drops older ones.  Per stream (models share
 * streams: an attached outlier forest runs on its parent's). */
struct RankWrites {
    uintptr_t p0, p1, l0, l1; /* proba [p0, p1), label [l0, l1) */
};
static std::mutex g_rank_writes_mu;
static std::unordered_map<cudaStream_t, std::deque<RankWrites>> g_rank_writes;

static bool rank_launch_pdl(cudaStream_t st, int sm_count, const void *rows, size_t rows_bytes, const void *proba, size_t psz, const int32_t *label,
                            int64_t n, int ostride) {
    static const bool no_pdl = getenv("B2F_NO_PDL") != nullptr;
    const int64_t ps = ostride & 0xffff, ls = (ostride >> 16) ? (ostride >> 16) : ps; /* ostride_p / ostride_l */
    RankWrites w;
    w.p0 = reinterpret_cast<uintptr_t>(proba);
    w.p1 = proba ? w.p0 + (size_t)((n - 1) * ps + 1) * psz : w.p0;
    w.l0 = reinterpret_cast<uintptr_t>(label);
    w.l1 = label ? w.l0 + (size_t)((n - 1) * ls + 1) * sizeof(int32_t) : w.l0;
    const uintptr_t r0 = reinterpret_cast<uintptr_t>(rows), r1 = r0 + rows_bytes;
    std::lock_guard<std::mutex> lk(g_rank_writes_mu);
    std::deque<RankWrites> &chain = g_rank_writes[st];
    bool pdl = !no_pdl;
    for (const RankWrites &c : chain)
        if ((c.p0 < r1 && r0 < c.p1) || (c.l0 < r1 && r0 < c.l1)) {
            pdl = false;
            break;
        }
    if (!pdl) chain.clear();
    chain.push_back(w);
    while (chain.size() > 2 * (size_t)sm_count + 1) chain.pop_front();
    return pdl;
}
static void rank_forget_stream(cudaStream_t st) {
    std::lock_guard<std::mutex> lk(g_rank_writes_mu);
    g_rank_writes.erase(st);
}

static int validate_blob(const uint8_t *blob, size_t nbytes, b2f_blob_header *hdr_out) {
    if (!blob || nbytes < sizeof(b2f_blob_header)) return set_err(B2F_EINVAL, "forest blob too small (%zu bytes)", nbytes);
    b2f_blob_header h;
    memcpy(&h, blob, sizeof(h));
    if (memcmp(h.magic, B2F_BLOB_MAGIC, 8) != 0) return set_err(B2F_EINVAL, "forest blob: bad magic");
    if (h.version != B2F_BLOB_VERSION) return set_err(B2F_EINVAL, "forest blob: version %u, expected %u", h.version, B2F_BLOB_VERSION);
    if (h.header_bytes != B2F_BLOB_HEADER_BYTES || h.row_words != B2F_ROW_WORDS)
        return set_err(B2F_EINVAL, "forest blob: header_bytes=%u row_words=%u unsupported", h.header_bytes, h.row_words);
    if (h.agg_mode != B2F_AGG_RF_MEAN && h.agg_mode != B2F_AGG_GBDT_LOGISTIC && h.agg_mode != B2F_AGG_IFOREST)
        return set_err(B2F_EINVAL, "forest blob: unknown agg_mode %u", h.agg_mode);
    if (h.n_trees == 0 || h.n_trees > B2F_MAX_TREES) return set_err(B2F_EINVAL, "forest blob: n_trees=%u out of range [1,%d]", h.n_trees, B2F_MAX_TREES);
    if (h.n_groups != (h.n_trees + 31) / 32) return set_err(B2F_EINVAL, "forest blob: n_groups=%u inconsistent with n_trees=%u", h.n_groups, h.n_trees);
    if (h.n_cat + h.n_num > B2F_SENTINEL_WORD) return set_err(B2F_EINVAL, "forest blob: n_cat+n_num=%u exceeds %u", h.n_cat + h.n_num, B2F_SENTINEL_WORD);
    if (h.total_bytes != nbytes) return set_err(B2F_EINVAL, "forest blob: total_bytes=%llu but %zu given", (unsigned long long)h.total_bytes, nbytes);
    if (h.groups_off < sizeof(h) || h.groups_off + (uint64_t)h.n_groups * sizeof(b2f_blob_group) > nbytes)
        return set_err(B2F_EINVAL, "forest blob: group table out of bounds");
    if (h.chunks_off % 256 || h.chunks_off + h.chunks_bytes > nbytes) return set_err(B2F_EINVAL, "forest blob: chunk area out of bounds");
    if (!(h.denom > 0.0)) return set_err(B2F_EINVAL, "forest blob: denom must be positive");
    const b2f_blob_group *gt = reinterpret_cast<const b2f_blob_group *>(blob + h.groups_off);
    uint64_t expect_off = 0;
    for (uint32_t g = 0; g < h.n_groups; ++g) {
        b2f_blob_group gr;
        memcpy(&gr, &gt[g], sizeof(gr));
        if (gr.chunk_off != expect_off || gr.n_slots == 0 || gr.n_leaf_slots == 0 ||
            gr.chunk_bytes != (gr.n_slots + gr.n_leaf_slots) * 256u || (uint64_t)gr.chunk_off + gr.chunk_bytes > h.chunks_bytes ||
            gr.n_slots >= (1u << 24) || gr.n_leaf_slots >= (1u << 24) || gr.n_trees == 0 || gr.n_trees > 32)
            return set_err(B2F_EINVAL, "forest blob: group %u descriptor invalid", g);
        expect_off += gr.chunk_bytes;
        /* every node word must keep the walk in bounds: check all slots */
        const uint32_t *N = reinterpret_cast<const uint32_t *>(blob + h.chunks_off + gr.chunk_off);
        for (uint32_t s = 0; s < gr.n_slots; ++s)
            for (uint32_t l = 0; l < 32; ++l) {
                const uint32_t t = N[(s * 32 + l) * 2], m = N[(s * 32 + l) * 2 + 1];
                const uint32_t feat = m >> B2F_META_FEAT_SHIFT, first = m & B2F_META_SLOT_MASK;
                const bool leaf = (first == s);
                if ((m & 0x03000000u) || feat > B2F_SENTINEL_WORD)
                    return set_err(B2F_EINVAL, "forest blob: group %u slot %u lane %u: bad meta word 0x%08x", g, s, l, m);
                if (leaf) {
                    if (!(m & B2F_META_CAT) || feat != B2F_SENTINEL_WORD || t >= gr.n_leaf_slots)
                        return set_err(B2F_EINVAL, "forest blob: group %u slot %u lane %u: malformed leaf", g, s, l);
                } else {
                    if (first <= s || first + 1 >= gr.n_slots) return set_err(B2F_EINVAL, "forest blob: group %u slot %u lane %u: child %u out of range", g, s, l, first);
                    if ((m & B2F_META_CAT) && feat >= h.n_cat && feat != B2F_SENTINEL_WORD)
                        return set_err(B2F_EINVAL, "forest blob: group %u slot %u lane %u: categorical test on numeric word", g, s, l);
                }
            }
    }
    if (expect_off != h.chunks_bytes) return set_err(B2F_EINVAL, "forest blob: chunks_bytes mismatch");
    *hdr_out = h;
    return B2F_OK;
}

extern "C" int b2f_blob_validate(const void *forest_blob, size_t nbytes) {
    b2f_blob_header h;
    return validate_blob(static_cast<const uint8_t *>(forest_blob), nbytes, &h);
}

/* ------------------------------------------------------------------ ranked rows: host-side tables (forest_rank.h) */
extern "C" b2f_ranker *b2f_ranker_create(const void *forest_blob, size_t nbytes) {
    b2f_blob_header h;
    if (validate_blob(static_cast<const uint8_t *>(forest_blob), nbytes, &h) != B2F_OK) return nullptr;
    b2f_ranker *r = new (std::nothrow) b2f_ranker();
    if (!r) {
        set_err(B2F_ENOMEM, "out of host memory");
        return nullptr;
    }
    ranker_build(r, static_cast<const uint8_t *>(forest_blob), h);
    return r;
}
extern "C" void b2f_ranker_destroy(b2f_ranker *r) { delete r; }

static void fill_rank_info(const b2f_ranker *r, bool ok, b2f_rank_info *out) {
    memset(out, 0, sizeof(*out));
    out->ok = ok ? 1 : 0;
    out->row_bytes = r->row_bytes;
    out->cat_bytes = r->cat_bytes;
    out->n_cat = r->n_cat;
    out->n_num = r->n_num;
    out->depth = r->depth;
    out->n_trees = r->n_trees;
    out->layout_bytes = (int32_t)r->layout.size();
    for (int j = 0; j < 16; ++j) {
        out->cat_shift[j] = r->cat_shift[j];
        out->cat_bits[j] = r->cat_bits[j];
    }
    for (size_t k = 0; k < r->thr.size() && k < 24; ++k) out->n_thresholds[k] = (int32_t)r->thr[k].size();
    out->n_pairs = (int32_t)r->pairs.size();
    for (size_t i = 0; i < r->pairs.size() && i < 128; ++i) out->pairs[i] = r->pairs[i];
    snprintf(out->why, sizeof(out->why), "%s", r->why);
}
extern "C" int b2f_ranker_info(const b2f_ranker *r, b2f_rank_info *out) {
    if (!r || !out) return set_err(B2F_EINVAL, "null argument");
    fill_rank_info(r, r->ok, out);
    return B2F_OK;
}
extern "C" const float *b2f_ranker_thresholds(const b2f_ranker *r, int k, int32_t *count) {
    if (!r || k < 0 || k >= (int)r->thr.size()) {
        if (count) *count = 0;
        return nullptr;
    }
    if (count) *count = (int32_t)r->thr[k].size();
    return r->thr[k].data();
}
extern "C" const void *b2f_ranker_layout(const b2f_ranker *r, int64_t *nbytes) {
    if (!r || !r->ok) {
        if (nbytes) *nbytes = 0;
        return nullptr;
    }
    if (nbytes) *nbytes = (int64_t)r->layout.size();
    return r->layout.data();
}
extern "C" int b2f_ranker_rank_rows(const b2f_ranker *r, const void *rows, int64_t n, int row_format, void *ranked_out, int threads) {
    if (!r || n < 0 || (n > 0 && (!rows || !ranked_out))) return set_err(B2F_EINVAL, "bad argument");
    if (!r->ok) return set_err(B2F_EINVAL, "no rank layout for this forest (%s)", r->why);
    if (row_format != B2F_ROWS_WORDS24 && row_format != B2F_ROWS_PACKED64) return set_err(B2F_EINVAL, "rows must be B2F_ROWS_WORDS24 or B2F_ROWS_PACKED64");
    if (row_format == B2F_ROWS_PACKED64 && !(r->n_cat == 9 && r->n_num <= 14)) return set_err(B2F_EINVAL, "schema does not fit the packed 64-byte row");
    threads = (int)std::min<int64_t>(std::max(threads, 1), std::max<int64_t>(1, n / 4096));
    const uint8_t *in = static_cast<const uint8_t *>(rows);
    uint8_t *out = static_cast<uint8_t *>(ranked_out);
    if (threads == 1) {
        rank_rows_range(r, in, 0, n, row_format, out);
        return B2F_OK;
    }
    std::vector<std::thread> pool;
    for (int t = 1; t < threads; ++t) pool.emplace_back([=] { rank_rows_range(r, in, n * t / threads, n * (t + 1) / threads, row_format, out); });
    rank_rows_range(r, in, 0, n / threads, row_format, out);
    for (auto &th : pool) th.join();
    return B2F_OK;
}

template <int R, bool SMEM, typename OutT>
static cudaError_t set_smem_attr(int bytes) {
    cudaError_t e = cudaFuncSetAttribute(k_forest_predict<R, SMEM, false, OutT>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(k_forest_predict<R, SMEM, true, OutT>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
}


/* ------------------------------------------------------------------ tile layout (forest_predict_tile.cuh)
 * Re-pack the interleaved blob tree-major: per tree its breadth-first nodes then its leaf payloads, trees in
 * U-groups of B2F_TILE_U (8) with an 80-byte descriptor, U-groups packed into pieces that fit a shared-memory ring slot. */
struct TileTree {
    std::vector<uint32_t> nodes; /* T, M pairs */
    std::vector<double> leaves;
    uint32_t depth = 0;
};

static bool extract_tree(const uint8_t *blob, const b2f_blob_header &h, const b2f_blob_group &gr, uint32_t lane, TileTree &out) {
    const uint32_t *N = reinterpret_cast<const uint32_t *>(blob + h.chunks_off + gr.chunk_off);
    const double *LV = reinterpret_cast<const double *>(blob + h.chunks_off + gr.chunk_off + (size_t)gr.n_slots * 256);
    std::vector<uint32_t> depth_of(gr.n_slots, 0);
    uint32_t reach = 0, max_leaf = 0, max_depth = 0;
    for (uint32_t s = 0; s <= reach; ++s) {
        const uint32_t t = N[(s * 32 + lane) * 2], m = N[(s * 32 + lane) * 2 + 1];
        const uint32_t feat = m >> B2F_META_FEAT_SHIFT, first = m & B2F_META_SLOT_MASK;
        const bool cat = (m & B2F_META_CAT) != 0;
        if (first >= B2F_TILE_MAX_TREE_NODES) return false;
        out.nodes.push_back(t);
        out.nodes.push_back((first << B2F_TILE_CHILD_SHIFT) | (cat ? B2F_TILE_META_CAT : 0u) | (feat << B2F_TILE_FEAT_SHIFT));
        if (first == s) { /* leaf */
            max_leaf = std::max(max_leaf, t);
            max_depth = std::max(max_depth, depth_of[s]);
        } else {
            reach = std::max(reach, first + 1);
            depth_of[first] = depth_of[first + 1] = depth_of[s] + 1;
        }
    }
    out.leaves.resize(max_leaf + 1);
    for (uint32_t i = 0; i <= max_leaf; ++i) out.leaves[i] = LV[i * 32 + lane];
    out.depth = max_depth;
    return true;
}

static bool build_tile_layout(const uint8_t *blob, const b2f_blob_header &h, uint32_t avail_smem, std::vector<uint8_t> &layout,
                              std::vector<TPiece> &pieces, uint32_t *slot_bytes, int *n_slots) {
    const b2f_blob_group *gt = reinterpret_cast<const b2f_blob_group *>(blob + h.groups_off);
    std::vector<TileTree> trees(h.n_trees);
    for (uint32_t t = 0; t < h.n_trees; ++t)
        if (!extract_tree(blob, h, gt[t / 32], t % 32, trees[t])) return false;
    /* U-groups */
    struct UG {
        uint32_t first, count, bytes;
    };
    std::vector<UG> ugs;
    uint64_t total = 0;
    for (uint32_t t = 0; t < h.n_trees; t += B2F_TILE_U) {
        UG u{t, std::min<uint32_t>(B2F_TILE_U, h.n_trees - t), (uint32_t)sizeof(TUGroup)};
        for (uint32_t k = 0; k < B2F_TILE_U; ++k)
            u.bytes += k < u.count ? (uint32_t)(trees[t + k].nodes.size() * 4 + trees[t + k].leaves.size() * 8) : 16u; /* stub: 1 node + 1 leaf */
        ugs.push_back(u);
        total += u.bytes;
    }
    /* piece size: if everything fits the ring, cut it into at most B2F_TILE_MAX_SLOTS pieces (resident: loaded
     * once per CTA, and walking starts when the first piece lands); otherwise ~32 KB pieces streamed through */
    uint32_t max_ug = 0;
    for (const UG &u : ugs) max_ug = std::max(max_ug, u.bytes);
    const bool fits = total + (uint64_t)(max_ug + 128) * B2F_TILE_MAX_SLOTS <= avail_smem;
    uint32_t target = fits ? (uint32_t)((total + B2F_TILE_MAX_SLOTS - 1) / B2F_TILE_MAX_SLOTS) + max_ug : 32u * 1024u;
    layout.clear();
    pieces.clear();
    size_t i = 0;
    uint32_t max_piece = 0;
    while (i < ugs.size()) {
        size_t j = i;
        uint32_t bytes = 0;
        while (j < ugs.size() && (j == i || bytes + ugs[j].bytes <= target)) bytes += ugs[j++].bytes;
        /* emit piece [i, j) */
        const uint32_t n_ug = (uint32_t)(j - i);
        const size_t start = layout.size();
        std::vector<uint8_t> buf((size_t)n_ug * sizeof(TUGroup));
        for (uint32_t g = 0; g < n_ug; ++g) {
            TUGroup d;
            memset(&d, 0, sizeof(d));
            for (uint32_t k = 0; k < B2F_TILE_U; ++k) {
                while (buf.size() % 8) buf.push_back(0);
                d.node_off[k] = (uint32_t)buf.size();
                if (k < ugs[i + g].count) {
                    const TileTree &tr = trees[ugs[i + g].first + k];
                    const uint8_t *np = reinterpret_cast<const uint8_t *>(tr.nodes.data());
                    buf.insert(buf.end(), np, np + tr.nodes.size() * 4);
                    d.leaf_off[k] = (uint32_t)buf.size();
                    const uint8_t *lp = reinterpret_cast<const uint8_t *>(tr.leaves.data());
                    buf.insert(buf.end(), lp, lp + tr.leaves.size() * 8);
                    d.depth = std::max(d.depth, tr.depth);
                } else { /* stub tree: one self-looping leaf worth 0.0 */
                    const uint32_t stub[2] = {0u, (0u << B2F_TILE_CHILD_SHIFT) | B2F_TILE_META_CAT | (B2F_SENTINEL_WORD << B2F_TILE_FEAT_SHIFT)};
                    const uint8_t *sp = reinterpret_cast<const uint8_t *>(stub);
                    buf.insert(buf.end(), sp, sp + 8);
                    d.leaf_off[k] = (uint32_t)buf.size();
                    const double z = 0.0;
                    const uint8_t *zp = reinterpret_cast<const uint8_t *>(&z);
                    buf.insert(buf.end(), zp, zp + 8);
                }
            }
            memcpy(buf.data() + (size_t)g * sizeof(TUGroup), &d, sizeof(d));
        }
        while (buf.size() % 128) buf.push_back(0);
        layout.insert(layout.end(), buf.begin(), buf.end());
        pieces.push_back(TPiece{(uint32_t)start, (uint32_t)buf.size(), n_ug, 0u});
        max_piece = std::max<uint32_t>(max_piece, (uint32_t)buf.size());
        i = j;
    }
    *slot_bytes = max_piece;
    if ((size_t)max_piece * pieces.size() <= avail_smem && pieces.size() <= B2F_TILE_MAX_SLOTS) {
        *n_slots = (int)pieces.size(); /* resident */
    } else {
        int s = (int)std::min<uint64_t>(B2F_TILE_MAX_SLOTS, avail_smem / max_piece);
        if (s < 2) return false; /* a single U-group does not fit a ring slot: tile kernel not applicable */
        *n_slots = s;
    }
    return true;
}

template <int D, int U, bool ST, typename OutT>
static cudaError_t rank_set_attr(int bytes) {
    return cudaFuncSetAttribute(k_forest_predict_rank<D, U, ST, OutT>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
}
template <int U, bool ST>
static cudaError_t rank_set_attr_all(int depth, int bytes) {
    cudaError_t e = cudaSuccess;
#define RK_ATTR(DD)                                                        \
    case DD:                                                               \
        e = rank_set_attr<DD, U, ST, float>(bytes);                        \
        if (e == cudaSuccess) e = rank_set_attr<DD, U, ST, double>(bytes); \
        break;
    switch (depth) {
        RK_ATTR(1) RK_ATTR(2) RK_ATTR(3) RK_ATTR(4) RK_ATTR(5) RK_ATTR(6) RK_ATTR(7) RK_ATTR(8)
        default: e = cudaErrorInvalidValue;
    }
#undef RK_ATTR
    return e;
}

static int rank_init(b2f_model *m, const uint8_t *blob) {
    m->rank_ok = false;
    ranker_build(&m->rk, blob, m->hdr);
    if (!m->rk.ok) return B2F_OK; /* no rank layout for this forest: the other kernels serve it */
    const char *off = getenv("B2F_RANK");
    if (off && !strcmp(off, "0")) return B2F_OK;
    const int64_t layout_bytes = (int64_t)m->rk.layout.size();
    /* resident: the per-group head table (rank_walk_group_head) follows the trees, 3U words per group of U trees */
    const int64_t head_bytes = (int64_t)m->rk.n_trees_padded * 12;
    const int64_t base = B2F_RANK_XS_BYTES /* alignment slack */ + (int64_t)B2F_RANK_PARTIALS * 32 * 8 + 256;
    int max_tiles = (int)std::min<int64_t>(B2F_RANK_MAX_TILES, ((int64_t)m->max_smem_optin - base - layout_bytes - head_bytes) / B2F_RANK_XS_BYTES);
    if (const char *mt = getenv("B2F_RANK_MAX_TILES")) max_tiles = std::min(max_tiles, std::max(1, atoi(mt)));
    /* resident while the whole layout fits next to a useful number of row tiles; otherwise it streams through a two-slot ring
     * in pieces of 8 trees (2 groups of 4: warp w owns (tile w / 2, group w mod 2), so <= 16 tiles per round) */
    m->rank_stream = max_tiles < 8;
    if (const char *fs = getenv("B2F_RANK_STREAM")) m->rank_stream = atoi(fs) != 0;
    int64_t forest_smem = layout_bytes + head_bytes;
    m->rank_u = 4;
    if (const char *ru = getenv("B2F_RANK_U")) m->rank_u = atoi(ru) == 8 ? 8 : 4;
    std::vector<uint8_t> dev_layout(m->rk.layout);
    if (m->rank_stream) {
        m->rank_u = 4;
        const int64_t piece = 8 * (int64_t)m->rk.tree_stride; /* n_trees_padded is a multiple of 8 */
        forest_smem = 2 * piece;
        max_tiles = (int)std::min<int64_t>(B2F_RANK_MAX_TILES, ((int64_t)m->max_smem_optin - base - forest_smem) / B2F_RANK_XS_BYTES);
        if (max_tiles < 4 || piece % 16) return B2F_OK;
    } else {
        const int U = m->rank_u, n_nodes = 1 << m->rk.depth;
        std::vector<uint32_t> head((size_t)head_bytes / 4, 0u);
        for (int t = 0; t < m->rk.n_trees_padded; ++t) {
            const uint32_t *nodes = reinterpret_cast<const uint32_t *>(m->rk.layout.data() + (size_t)t * m->rk.tree_stride);
            uint32_t *g = head.data() + (size_t)(t / U) * 3 * U;
            g[t % U] = nodes[0];
            if (n_nodes > 2) { /* depth 1: no level 1 (node word 1 is the unused last one) */
                g[U + 2 * (t % U)] = nodes[1];
                g[U + 2 * (t % U) + 1] = nodes[2];
            }
        }
        dev_layout.resize((size_t)(layout_bytes + head_bytes));
        memcpy(dev_layout.data() + layout_bytes, head.data(), (size_t)head_bytes);
    }
    CUDA_TRY(cudaMalloc(&m->d_rank_layout, dev_layout.size()));
    CUDA_TRY(cudaMemcpy(m->d_rank_layout, dev_layout.data(), dev_layout.size(), cudaMemcpyHostToDevice));
    RParams &rp = m->rp;
    memset(&rp, 0, sizeof(rp));
    rp.layout = static_cast<const uint8_t *>(m->d_rank_layout);
    rp.layout_bytes = (uint32_t)dev_layout.size();
    rp.tree_stride = m->rk.tree_stride;
    rp.n_trees_padded = m->rk.n_trees_padded;
    rp.n_groups = (m->rk.n_trees + m->rank_u - 1) / m->rank_u;
    rp.head_off = (uint32_t)layout_bytes;
    rp.depth = m->rk.depth;
    rp.agg_mode = (int)m->hdr.agg_mode;
    rp.n_cat = m->rk.n_cat;
    rp.n_num = m->rk.n_num;
    rp.row_bytes = m->rk.row_bytes;
    rp.cat_bytes = m->rk.cat_bytes;
    rp.max_tiles = max_tiles;
    rp.groups_per_piece = 2;
    rp.piece_bytes = 8u * m->rk.tree_stride;
    rp.n_pieces = m->rk.n_trees_padded / 8;
    rp.init_raw = m->hdr.init_raw;
    rp.denom = m->hdr.denom;
    rp.threshold = m->hdr.threshold;
    rp.mul_two = 2u;
    rp.mul_64k = 65536u;
    rp.add_64k = 65535u;
    rp.n_pairs = (int)m->rk.pairs.size();
    for (int j = 0; j < 16; ++j) {
        rp.cat_shift[j] = (uint8_t)m->rk.cat_shift[j];
        rp.cat_bits[j] = (uint8_t)m->rk.cat_bits[j];
        rp.cat_start[j] = 0;
        rp.cat_mask[j] = 0ull;
    }
    for (int i = rp.n_pairs - 1; i >= 0; --i) { /* pairs are sorted by (feature, category): the last write per feature is its first pair */
        const uint32_t j = m->rk.pairs[i] >> 16, c = m->rk.pairs[i] & 0xFFFFu;
        rp.cat_start[j] = (uint8_t)i;
        rp.cat_mask[j] |= 1ull << c;
    }
#ifdef B2F_RANK_TRACE
    const size_t trace_bytes = (size_t)B2F_RANK_TRACE_LAUNCHES * m->sm_count * B2F_RANK_TRACE_WORDS * sizeof(unsigned long long);
    CUDA_TRY(cudaMalloc(&m->d_rank_trace, trace_bytes));
    CUDA_TRY(cudaMemset(m->d_rank_trace, 0, trace_bytes));
#endif
    m->rank_smem_bytes = (int)(B2F_RANK_XS_BYTES + (int64_t)max_tiles * B2F_RANK_XS_BYTES + (int64_t)B2F_RANK_PARTIALS * 32 * 8 + forest_smem);
    if (m->rank_stream)
        CUDA_TRY((rank_set_attr_all<4, true>(rp.depth, m->rank_smem_bytes)));
    else
        CUDA_TRY(m->rank_u == 8 ? (rank_set_attr_all<8, false>(rp.depth, m->rank_smem_bytes)) : (rank_set_attr_all<4, false>(rp.depth, m->rank_smem_bytes)));
    m->rank_ok = true;
    return B2F_OK;
}

static bool kn_env_is(const char *v) {
    const char *kn = getenv("B2F_KERNEL");
    return kn && !strcmp(kn, v);
}

static int model_init_cuda(b2f_model *m, const uint8_t *blob, size_t nbytes) {
    CUDA_TRY(cudaSetDevice(m->device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, m->device));
    if (prop.major < 10)
        return set_err(B2F_ENODEV, "device %d is sm_%d%d; this library is built for sm_100a (B200) only", m->device, prop.major, prop.minor);
    m->sm_count = prop.multiProcessorCount;
    CUDA_TRY(cudaDeviceGetAttribute(&m->max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, m->device));

    CUDA_TRY(cudaMalloc(&m->d_blob, nbytes));
    CUDA_TRY(cudaMemcpy(m->d_blob, blob, nbytes, cudaMemcpyHostToDevice));
    m->forest_bytes = (int64_t)m->hdr.chunks_bytes;

    KParams &kp = m->kp;
    memset(&kp, 0, sizeof(kp));
    kp.chunks = static_cast<const uint8_t *>(m->d_blob) + m->hdr.chunks_off;
    kp.n_groups = (int)m->hdr.n_groups;
    kp.agg_mode = (int)m->hdr.agg_mode;
    kp.n_cat = (int)m->hdr.n_cat;
    kp.n_num = (int)m->hdr.n_num;
    kp.init_raw = m->hdr.init_raw;
    kp.denom = m->hdr.denom;
    kp.threshold = m->hdr.threshold;
    memcpy(kp.impute, m->hdr.impute, sizeof(kp.impute));
    const b2f_blob_group *gt = reinterpret_cast<const b2f_blob_group *>(blob + m->hdr.groups_off);
    for (uint32_t g = 0; g < m->hdr.n_groups; ++g) {
        kp.g[g].chunk_off = gt[g].chunk_off;
        kp.g[g].chunk_bytes = gt[g].chunk_bytes;
        kp.g[g].n_slots = gt[g].n_slots;
        kp.g[g].n_leaf_slots = gt[g].n_leaf_slots;
        kp.g[g].depth = gt[g].depth;
    }

    /* the packed 64-byte row needs the credit-default shape: exactly 9 categoricals of <= 126 categories, <= 14 numerics */
    m->packed_ok = m->hdr.n_cat == 9 && m->hdr.n_num <= 14; /* the kernels decode word L-7 / q[2+k] for exactly nine 7-bit fields */
    for (uint32_t f = 0; f < m->hdr.n_cat; ++f)
        if (m->hdr.vocab[f] > 126) m->packed_ok = false;

    /* shared-memory residency: whole forest + static barriers must fit the opt-in limit */
    const int64_t need = (int64_t)m->hdr.chunks_bytes;
    const char *force = getenv("B2F_FORCE_WALK"); /* "smem" | "global": test hook */
    bool fits = need + 1024 <= (int64_t)m->max_smem_optin;
    if (force && !strcmp(force, "global")) fits = false;
    if (force && !strcmp(force, "smem") && !fits) return set_err(B2F_EINVAL, "B2F_FORCE_WALK=smem but forest needs %lld bytes", (long long)need);
    m->walk_mode = fits ? B2F_WALK_SMEM : B2F_WALK_GLOBAL;
    m->smem_bytes = fits ? (int)need : 0;
    if (fits) {
        CUDA_TRY((set_smem_attr<1, true, float>(m->smem_bytes)));
        CUDA_TRY((set_smem_attr<2, true, float>(m->smem_bytes)));
        CUDA_TRY((set_smem_attr<4, true, float>(m->smem_bytes)));
        CUDA_TRY((set_smem_attr<1, true, double>(m->smem_bytes)));
        CUDA_TRY((set_smem_attr<2, true, double>(m->smem_bytes)));
        CUDA_TRY((set_smem_attr<4, true, double>(m->smem_bytes)));
    }
    const char *cr = getenv("B2F_CHUNK_ROWS"); /* tuning hook: rows per pipelined H2D/kernel/D2H chunk */
    if (cr && atoll(cr) >= 1024) m->chunk_rows = atoll(cr);
    m->chunk_plan = {768}; /* measured best on B200 for 65 536-row batches: 3/4 of the batch, then the rest */
    if (const char *pl = getenv("B2F_CHUNK_PLAN")) {
        m->chunk_plan.clear();
        for (const char *q = pl; *q;) {
            m->chunk_plan.push_back(atoll(q));
            while (*q && *q != ',') ++q;
            if (*q == ',') ++q;
        }
    }
    /* latency kernel: while rows x groups warps still fit about two waves of the chip */
    /* the latency form (one CTA per 2 rows, warp = tree group) hands over to the warp-per-row kernel at 3 072 rows: measured on
     * B200 (profiles/r02_split_threshold.json, synchronous 64-byte-row calls) it is never slower below that -- GBDT 500 x d8:
     * 35 vs 60 us at 1 024 rows, 59 vs 71 at 3 072, equal at 4 096; GBDT 100 x d6: equal from 512 rows up.  (Round 1 scaled the
     * threshold with the number of tree groups: 592 rows for 500 trees, which left 768..3 072-row requests on the slower kernel.) */
    m->split_max_rows = 3072;
    if (const char *sp = getenv("B2F_SPLIT_MAX_ROWS")) m->split_max_rows = atoll(sp);
    if (kn_env_is("warp") || kn_env_is("tile")) m->split_max_rows = 0; /* tests pin one kernel */
    if (kn_env_is("split")) m->split_max_rows = INT64_MAX;
    const char *rpw = getenv("B2F_ROWS_PER_WARP");
    m->rows_per_warp_max = 2;
    if (rpw) {
        int v = atoi(rpw);
        if (v == 1 || v == 2 || v == 4) m->rows_per_warp_max = v;
    }

    /* tile kernel: tree-major layout + shared-memory ring plan */
    {
        const char *kn = getenv("B2F_KERNEL"); /* "warp" | "tile" | unset = choose by batch size */
        const char *tm = getenv("B2F_TILE_MIN_ROWS");
        std::vector<uint8_t> layout;
        std::vector<TPiece> pieces;
        uint32_t slot_bytes = 0;
        int n_slots = 0;
        bool ok = false;
        /* most consumer warps for which the forest still stays resident; else 16 warps and a streamed forest */
        int cwarps = B2F_TILE_WARPS_MIN;
        if (!(kn && !strcmp(kn, "warp"))) {
            if (const char *tw = getenv("B2F_TILE_WARPS")) {
                cwarps = std::min(B2F_TILE_WARPS_MAX, std::max(1, atoi(tw)));
                const uint32_t avail = (uint32_t)m->max_smem_optin - 1024u - 4096u - (uint32_t)cwarps * B2F_TILE_XS_BYTES;
                ok = build_tile_layout(blob, m->hdr, avail, layout, pieces, &slot_bytes, &n_slots);
            } else {
                for (int w = B2F_TILE_WARPS_MAX; w >= B2F_TILE_WARPS_MIN && !ok; w -= 4) {
                    const uint32_t avail = (uint32_t)m->max_smem_optin - 1024u - 4096u - (uint32_t)w * B2F_TILE_XS_BYTES;
                    const bool built = build_tile_layout(blob, m->hdr, avail, layout, pieces, &slot_bytes, &n_slots);
                    const bool res = built && (int)pieces.size() <= n_slots;
                    if (built && (res || w == B2F_TILE_WARPS_MIN)) {
                        ok = true;
                        cwarps = w;
                    }
                }
            }
        }
        if (ok) {
            CUDA_TRY(cudaMalloc(&m->d_tile_layout, layout.size()));
            CUDA_TRY(cudaMemcpy(m->d_tile_layout, layout.data(), layout.size(), cudaMemcpyHostToDevice));
            CUDA_TRY(cudaMalloc((void **)&m->d_tile_pieces, pieces.size() * sizeof(TPiece)));
            CUDA_TRY(cudaMemcpy(m->d_tile_pieces, pieces.data(), pieces.size() * sizeof(TPiece), cudaMemcpyHostToDevice));
            TParams &tp = m->tp;
            memset(&tp, 0, sizeof(tp));
            tp.layout = static_cast<const uint8_t *>(m->d_tile_layout);
            tp.pieces = m->d_tile_pieces;
            tp.n_pieces = (int)pieces.size();
            tp.n_slots = n_slots;
            tp.slot_bytes = slot_bytes;
            tp.agg_mode = kp.agg_mode;
            tp.n_cat = kp.n_cat;
            tp.n_num = kp.n_num;
            tp.init_raw = kp.init_raw;
            tp.denom = kp.denom;
            tp.threshold = kp.threshold;
            memcpy(tp.impute, kp.impute, sizeof(tp.impute));
            m->tile_cwarps = cwarps;
            m->tile_smem_bytes = 4096 + cwarps * B2F_TILE_XS_BYTES + n_slots * (int)slot_bytes;
            m->tile_layout_bytes = (int64_t)layout.size();
            CUDA_TRY(cudaFuncSetAttribute(k_forest_predict_tile<false, float>, cudaFuncAttributeMaxDynamicSharedMemorySize, m->tile_smem_bytes));
            CUDA_TRY(cudaFuncSetAttribute(k_forest_predict_tile<false, double>, cudaFuncAttributeMaxDynamicSharedMemorySize, m->tile_smem_bytes));
            CUDA_TRY(cudaFuncSetAttribute(k_forest_predict_tile<true, float>, cudaFuncAttributeMaxDynamicSharedMemorySize, m->tile_smem_bytes));
            CUDA_TRY(cudaFuncSetAttribute(k_forest_predict_tile<true, double>, cudaFuncAttributeMaxDynamicSharedMemorySize, m->tile_smem_bytes));
            m->tile_ok = true;
            /* crossover measured on B200 (tools/ksweep.py): a resident forest ties with the warp kernel from
             * 65 536 rows up (and sums in sklearn's tree order); a streamed forest wins from ~24k rows */
            m->tile_min_rows = (tp.n_pieces <= tp.n_slots) ? 65536 : 24576;
            if (tm && atoll(tm) >= 0) m->tile_min_rows = atoll(tm);
            if (kn && !strcmp(kn, "tile")) m->tile_min_rows = 1;
        } else if (kn && !strcmp(kn, "tile")) {
            return set_err(B2F_EINVAL, "B2F_KERNEL=tile but the forest's trees do not fit the tile kernel's shared-memory ring");
        }
    }

    /* rank kernel: 4-byte integer nodes, complete trees, rows as ranks (forest_rank.h); only while the layout stays resident */
    {
        int rc = rank_init(m, blob);
        if (rc) return rc;
    }

    for (int s = 0; s < B2F_STREAMS; ++s) CUDA_TRY(cudaStreamCreateWithFlags(&m->slots[s].stream, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&m->compute, cudaStreamNonBlocking));

    CUDA_TRY(cudaFuncSetAttribute(k_feature_moments, cudaFuncAttributeMaxDynamicSharedMemorySize, B2F_MOM_SMEM));
    m->mom_blocks = m->sm_count * 3; /* one full wave: 3 CTAs (3-stage 72 KB ring each) per SM */
    CUDA_TRY(cudaMalloc(&m->d_mom_partials, (size_t)m->mom_blocks * B2F_MOM_VALUES * sizeof(double)));
    CUDA_TRY(cudaMalloc(&m->d_mom_ticket, sizeof(unsigned int)));
    CUDA_TRY(cudaMemset(m->d_mom_ticket, 0, sizeof(unsigned int)));
    CUDA_TRY(cudaMalloc(&m->d_mom_out, B2F_MOM_VALUES * sizeof(double)));
    return B2F_OK;
}

extern "C" b2f_model *b2f_model_create(const void *forest_blob, size_t nbytes, int device) {
    int ndev = b2f_device_count();
    if (ndev < 0) return nullptr;
    if (device < 0 || device >= ndev) {
        set_err(B2F_EINVAL, "device %d out of range (have %d)", device, ndev);
        return nullptr;
    }
    b2f_model *m = new (std::nothrow) b2f_model();
    if (!m) {
        set_err(B2F_ENOMEM, "out of host memory");
        return nullptr;
    }
    m->device = device;
    if (validate_blob(static_cast<const uint8_t *>(forest_blob), nbytes, &m->hdr) != B2F_OK ||
        model_init_cuda(m, static_cast<const uint8_t *>(forest_blob), nbytes) != B2F_OK) {
        char keep[sizeof(g_err)];
        memcpy(keep, g_err, sizeof(keep));
        b2f_model_destroy(m);
        memcpy(g_err, keep, sizeof(keep));
        return nullptr;
    }
    return m;
}

extern "C" void b2f_model_destroy(b2f_model *m) {
    if (!m) return;
    cudaSetDevice(m->device);
    cudaDeviceSynchronize();
    if (m->outlier) b2f_model_destroy(m->outlier);
    if (m->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(m->comm);
    for (int s = 0; s < B2F_STREAMS; ++s) {
        Slot &sl = m->slots[s];
        if (sl.d_rows) cudaFree(sl.d_rows);
        if (sl.d_proba) cudaFree(sl.d_proba);
        if (sl.d_label) cudaFree(sl.d_label);
        if (sl.stream) {
            rank_forget_stream(sl.stream);
            cudaStreamDestroy(sl.stream);
        }
    }
    for (auto &t : m->tickets)
        for (auto &e : t.ev)
            if (e) cudaEventDestroy(e);
    if (m->compute) {
        rank_forget_stream(m->compute);
        cudaStreamDestroy(m->compute);
    }
    if (m->d_blob) cudaFree(m->d_blob);
    if (m->d_tile_layout) cudaFree(m->d_tile_layout);
    if (m->d_tile_pieces) cudaFree(m->d_tile_pieces);
    if (m->d_rank_layout) cudaFree(m->d_rank_layout);
#ifdef B2F_RANK_TRACE
    if (m->d_rank_trace) cudaFree(m->d_rank_trace);
#endif
    if (m->d_mom_rows) cudaFree(m->d_mom_rows);
    if (m->d_mom_partials) cudaFree(m->d_mom_partials);
    if (m->d_mom_ticket) cudaFree(m->d_mom_ticket);
    if (m->d_mom_out) cudaFree(m->d_mom_out);
    if (m->d_gather) cudaFree(m->d_gather);
    if (m->d_flush) cudaFree(m->d_flush);
    delete m;
}

static int pick_rows_per_warp(const b2f_model *m, int64_t n) {
    int r = m->rows_per_warp_max;
    const int64_t warps = (int64_t)m->sm_count * B2F_PREDICT_WARPS;
    while (r > 1 && n / r < warps) r >>= 1; /* small batches: spread rows over more warps */
    return r;
}

extern "C" int b2f_model_info(const b2f_model *m, b2f_info *out) {
    if (!m || !out) return set_err(B2F_EINVAL, "null argument");
    memset(out, 0, sizeof(*out));
    out->device = m->device;
    out->sm_count = m->sm_count;
    out->agg_mode = (int)m->hdr.agg_mode;
    out->walk_mode = m->walk_mode;
    out->n_trees = (int)m->hdr.n_trees;
    out->n_groups = (int)m->hdr.n_groups;
    out->max_depth = (int)m->hdr.max_depth;
    out->n_cat = (int)m->hdr.n_cat;
    out->n_num = (int)m->hdr.n_num;
    out->smem_bytes = m->smem_bytes;
    out->block_threads = B2F_PREDICT_THREADS;
    out->rows_per_warp = m->rows_per_warp_max;
    out->forest_bytes = m->forest_bytes;
    out->launches = m->launches + (m->outlier ? m->outlier->launches : 0);
    out->launches_tile = m->launches_tile + (m->outlier ? m->outlier->launches_tile : 0);
    out->tile_min_rows = m->tile_min_rows;
    out->tile_ok = m->tile_ok ? 1 : 0;
    out->tile_resident = (m->tile_ok && m->tp.n_pieces <= m->tp.n_slots) ? 1 : 0;
    out->packed_ok = m->packed_ok ? 1 : 0;
    out->tile_warps = m->tile_ok ? m->tile_cwarps : 0;
    out->launches_split = m->launches_split;
    out->split_max_rows = m->split_max_rows;
    out->outlier_trees = m->outlier ? (int)m->outlier->hdr.n_trees : 0;
    out->rank_ok = m->rank_ok ? 1 : 0;
    out->launches_rank = m->launches_rank;
    out->rank_smem_bytes = m->rank_ok ? m->rank_smem_bytes : 0;
    out->rank_row_bytes = m->rk.row_bytes;
    out->rank_stream = (m->rank_ok && m->rank_stream) ? 1 : 0;
    out->rank_last_pdl = m->rank_last_pdl ? 1 : 0;
    return B2F_OK;
}

extern "C" int b2f_model_rank_info(const b2f_model *m, b2f_rank_info *out) {
    if (!m || !out) return set_err(B2F_EINVAL, "null argument");
    fill_rank_info(&m->rk, m->rank_ok, out);
    if (m->rk.ok && !m->rank_ok) snprintf(out->why, sizeof(out->why), "the rank layout (%zu bytes) does not stay resident in shared memory", m->rk.layout.size());
    return B2F_OK;
}

/* ------------------------------------------------------------------ pinned memory */
extern "C" void *b2f_pinned_alloc(size_t nbytes) {
    void *p = nullptr;
    cudaError_t e = cudaHostAlloc(&p, nbytes ? nbytes : 1, cudaHostAllocPortable);
    if (e != cudaSuccess) {
        set_err(B2F_ENOMEM, "cudaHostAlloc(%zu) failed: %s", nbytes, cudaGetErrorString(e));
        return nullptr;
    }
    return p;
}
extern "C" void b2f_pinned_free(void *p) {
    if (p) cudaFreeHost(p);
}

/* ------------------------------------------------------------------ kernel launch */
template <int R, bool SMEM, bool PACKED, typename OutT>
static cudaError_t launch_one(const b2f_model *m, cudaStream_t st, const void *rows, int64_t n, void *proba, int32_t *label, int ostride) {
    const int64_t n_batches = (n + R - 1) / R;
    int64_t ctas = std::min<int64_t>(m->sm_count, n_batches);
    if (ctas < 1) ctas = 1;
    k_forest_predict<R, SMEM, PACKED, OutT><<<(unsigned)ctas, B2F_PREDICT_THREADS, SMEM ? m->smem_bytes : 0, st>>>(
        m->kp, static_cast<const uint32_t *>(rows), (long long)n, static_cast<OutT *>(proba), label, ostride);
    return cudaGetLastError();
}

template <bool PACKED, typename OutT>
static cudaError_t launch_tile(const b2f_model *m, cudaStream_t st, const void *rows, int64_t n, void *proba, int32_t *label, int ostride) {
    const int64_t n_tiles = (n + B2F_TILE_ROWS - 1) / B2F_TILE_ROWS;
    const unsigned ctas = (unsigned)std::max<int64_t>(1, std::min<int64_t>(m->sm_count, n_tiles));
    k_forest_predict_tile<PACKED, OutT><<<ctas, (unsigned)(m->tile_cwarps + 1) * 32u, m->tile_smem_bytes, st>>>(m->tp, static_cast<const uint32_t *>(rows), (long long)n,
                                                                                           static_cast<OutT *>(proba), label, ostride);
    return cudaGetLastError();
}

template <bool PACKED, typename OutT>
static cudaError_t launch_split(const b2f_model *m, cudaStream_t st, const void *rows, int64_t n, void *proba, int32_t *label, int ostride) {
    constexpr int R = 2;
    const unsigned ctas = (unsigned)((n + R - 1) / R);
    k_forest_predict_split<R, PACKED, OutT><<<ctas, 32u * (unsigned)m->kp.n_groups, 0, st>>>(m->kp, static_cast<const uint32_t *>(rows), (long long)n,
                                                                                            static_cast<OutT *>(proba), label, ostride);
    return cudaGetLastError();
}

/* the rank kernel goes out with programmatic stream serialization (see rank_launch_pdl) */
template <int D, int U, bool ST, typename OutT>
static cudaError_t launch_rank_du(const b2f_model *m, cudaStream_t st, const void *rows, int64_t n, void *proba, int32_t *label, int ostride, bool pdl) {
    const int64_t n_tiles = (n + 31) / 32;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)std::max<int64_t>(1, std::min<int64_t>(m->sm_count, n_tiles)));
    cfg.blockDim = dim3(B2F_RANK_THREADS);
    cfg.dynamicSmemBytes = (size_t)m->rank_smem_bytes;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
#ifdef B2F_RANK_TRACE
    RParams rp = m->rp; /* launch i records into slot i mod B2F_RANK_TRACE_LAUNCHES */
    rp.trace = m->d_rank_trace + (size_t)(m->launches_rank % B2F_RANK_TRACE_LAUNCHES) * m->sm_count * B2F_RANK_TRACE_WORDS;
#else
    const RParams &rp = m->rp;
#endif
    return cudaLaunchKernelEx(&cfg, k_forest_predict_rank<D, U, ST, OutT>, rp, static_cast<const uint8_t *>(rows), (long long)n,
                              static_cast<OutT *>(proba), label, ostride);
}

#ifdef B2F_RANK_TRACE
/* traced build only: copy the trace ring (B2F_RANK_TRACE_LAUNCHES x sm_count x B2F_RANK_TRACE_WORDS words) to the host after
 * a synchronise; returns the rank launches made so far (launch i sits in slot i mod B2F_RANK_TRACE_LAUNCHES) */
extern "C" int64_t b2f_rank_trace_read(b2f_model *m, unsigned long long *out, int32_t *launch_slots, int32_t *ctas_per_launch) {
    if (!m || !out || !m->d_rank_trace) return -1;
    if (cudaSetDevice(m->device) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess) return -1;
    if (cudaMemcpy(out, m->d_rank_trace, (size_t)B2F_RANK_TRACE_LAUNCHES * m->sm_count * B2F_RANK_TRACE_WORDS * sizeof(unsigned long long),
                   cudaMemcpyDeviceToHost) != cudaSuccess)
        return -1;
    *launch_slots = B2F_RANK_TRACE_LAUNCHES;
    *ctas_per_launch = m->sm_count;
    return m->launches_rank;
}
#endif
template <typename OutT>
static cudaError_t launch_rank(const b2f_model *m, cudaStream_t st, const void *rows, int64_t n, void *proba, int32_t *label, int ostride, bool pdl) {
#define RK_CASE(DD)                                                                                                  \
    case DD:                                                                                                         \
        if (m->rank_stream) return launch_rank_du<DD, 4, true, OutT>(m, st, rows, n, proba, label, ostride, pdl);     \
        return m->rank_u == 8 ? launch_rank_du<DD, 8, false, OutT>(m, st, rows, n, proba, label, ostride, pdl)        \
                              : launch_rank_du<DD, 4, false, OutT>(m, st, rows, n, proba, label, ostride, pdl);
    switch (m->rp.depth) {
        RK_CASE(1) RK_CASE(2) RK_CASE(3) RK_CASE(4) RK_CASE(5) RK_CASE(6) RK_CASE(7) RK_CASE(8)
    }
#undef RK_CASE
    return cudaErrorInvalidValue;
}

static size_t row_bytes_of(const b2f_model *m, int fmt) {
    return fmt == B2F_ROWS_RANKED ? (size_t)m->rk.row_bytes : (fmt == B2F_ROWS_PACKED64 ? B2F_PACKED_ROW_BYTES : B2F_ROW_BYTES);
}

static int check_row_format(const b2f_model *m, int fmt) {
    if (fmt == B2F_ROWS_WORDS24) return B2F_OK;
    if (fmt == B2F_ROWS_RANKED) {
        if (!m->rank_ok)
            return set_err(B2F_EINVAL, "B2F_ROWS_RANKED is not available for this model (%s)",
                           m->rk.ok ? "its rank layout fits neither shared memory nor the streaming ring" : m->rk.why);
        return B2F_OK;
    }
    if (fmt != B2F_ROWS_PACKED64) return set_err(B2F_EINVAL, "unknown row format %d", fmt);
    if (!m->packed_ok) return set_err(B2F_EINVAL, "this model's schema does not fit the packed 64-byte row (needs exactly 9 categoricals with <= 126 categories, <= 14 numerics)");
    return B2F_OK;
}

static int launch_predict(b2f_model *m, cudaStream_t st, const void *rows_dev, int64_t n, int fmt, void *proba_dev, int f64, int32_t *label_dev,
                          int ostride = 1) {
    if (n <= 0) return B2F_OK;
    const bool pk = fmt == B2F_ROWS_PACKED64;
    cudaError_t e;
    if (fmt == B2F_ROWS_RANKED) { /* ranked rows have one kernel: integer compares on the resident rank layout */
        const bool pdl = rank_launch_pdl(st, m->sm_count, rows_dev, (size_t)n * (size_t)m->rk.row_bytes, proba_dev, f64 ? sizeof(double) : sizeof(float), label_dev, n, ostride);
        e = f64 ? launch_rank<double>(m, st, rows_dev, n, proba_dev, label_dev, ostride, pdl)
                : launch_rank<float>(m, st, rows_dev, n, proba_dev, label_dev, ostride, pdl);
        if (e != cudaSuccess) return set_err(B2F_ECUDA, "k_forest_predict_rank launch failed: %s", cudaGetErrorString(e));
        m->launches++;
        m->launches_rank++;
        m->rank_last_pdl = pdl;
        return B2F_OK;
    }
    if (m->tile_ok && n >= m->tile_min_rows) {
        e = pk ? (f64 ? launch_tile<true, double>(m, st, rows_dev, n, proba_dev, label_dev, ostride) : launch_tile<true, float>(m, st, rows_dev, n, proba_dev, label_dev, ostride))
               : (f64 ? launch_tile<false, double>(m, st, rows_dev, n, proba_dev, label_dev, ostride) : launch_tile<false, float>(m, st, rows_dev, n, proba_dev, label_dev, ostride));
        if (e != cudaSuccess) return set_err(B2F_ECUDA, "k_forest_predict_tile launch failed: %s", cudaGetErrorString(e));
        m->launches++;
        m->launches_tile++;
        return B2F_OK;
    }
    if (n <= m->split_max_rows) { /* a handful of rows: spread each row's tree groups over the warps of a CTA */
        e = pk ? (f64 ? launch_split<true, double>(m, st, rows_dev, n, proba_dev, label_dev, ostride) : launch_split<true, float>(m, st, rows_dev, n, proba_dev, label_dev, ostride))
               : (f64 ? launch_split<false, double>(m, st, rows_dev, n, proba_dev, label_dev, ostride) : launch_split<false, float>(m, st, rows_dev, n, proba_dev, label_dev, ostride));
        if (e != cudaSuccess) return set_err(B2F_ECUDA, "k_forest_predict_split launch failed: %s", cudaGetErrorString(e));
        m->launches++;
        m->launches_split++;
        return B2F_OK;
    }
    const int r = pick_rows_per_warp(m, n);
    const bool sm = m->walk_mode == B2F_WALK_SMEM;
#define DISPATCH_T(RR, SM, PK)                                                                                      \
    (f64 ? launch_one<RR, SM, PK, double>(m, st, rows_dev, n, proba_dev, label_dev, ostride)                         \
         : launch_one<RR, SM, PK, float>(m, st, rows_dev, n, proba_dev, label_dev, ostride))
#define DISPATCH(RR) (sm ? (pk ? DISPATCH_T(RR, true, true) : DISPATCH_T(RR, true, false)) : (pk ? DISPATCH_T(RR, false, true) : DISPATCH_T(RR, false, false)))
    if (r == 4)
        e = DISPATCH(4);
    else if (r == 2)
        e = DISPATCH(2);
    else
        e = DISPATCH(1);
#undef DISPATCH
#undef DISPATCH_T
    if (e != cudaSuccess) return set_err(B2F_ECUDA, "k_forest_predict launch failed: %s", cudaGetErrorString(e));
    m->launches++;
    return B2F_OK;
}

/* ------------------------------------------------------------------ host-buffer pipeline */
static int slot_reserve(b2f_model *m, Slot &sl, int64_t rows) {
    if (rows <= sl.cap_rows) return B2F_OK;
    CUDA_TRY(cudaStreamSynchronize(sl.stream));
    if (sl.d_rows) cudaFree(sl.d_rows);
    if (sl.d_proba) cudaFree(sl.d_proba);
    if (sl.d_label) cudaFree(sl.d_label);
    sl.d_rows = sl.d_proba = nullptr;
    sl.d_label = nullptr;
    sl.cap_rows = 0;
    int64_t cap = std::max<int64_t>(rows, 1024);
    CUDA_TRY(cudaMalloc(&sl.d_rows, (size_t)cap * B2F_ROW_BYTES));
    CUDA_TRY(cudaMalloc(&sl.d_proba, (size_t)cap * sizeof(b2f_scored_full)));
    CUDA_TRY(cudaMalloc((void **)&sl.d_label, (size_t)cap * sizeof(int32_t)));
    sl.cap_rows = cap;
    return B2F_OK;
}

/* enqueue the whole batch; on return used_mask tells which slot streams carry work.
 * B2F_TIMELINE=1 (debug): record an event after every operation and print the schedule to stderr. */
static int enqueue_host_batch(b2f_model *m, const void *rows, int64_t n, int fmt, void *proba, int f64, int32_t *label, uint32_t *used_mask) {
    *used_mask = 0;
    if (n < 0) return set_err(B2F_EINVAL, "negative row count");
    if (n == 0) return B2F_OK;
    if (!rows) return set_err(B2F_EINVAL, "rows is NULL");
    {
        int rcf = check_row_format(m, fmt);
        if (rcf) return rcf;
    }
    const size_t row_bytes = row_bytes_of(m, fmt);
    CUDA_TRY(cudaSetDevice(m->device));
    int64_t chunk = m->chunk_rows;
    if (n <= chunk + chunk / 2) chunk = n; /* small batch: one H2D, one launch */
    const size_t psz = f64 == 1 ? sizeof(double) : sizeof(float);
    static const bool timeline = getenv("B2F_TIMELINE") != nullptr;
    std::vector<cudaEvent_t> tev;
    auto mark = [&](cudaStream_t st) {
        if (!timeline) return;
        cudaEvent_t e;
        cudaEventCreate(&e);
        cudaEventRecord(e, st);
        tev.push_back(e);
    };
    /* chunk schedule: equal chunks by default; a plan (B2F_CHUNK_PLAN="a,b,c": fractions of the batch in
     * 1/1024ths, the last chunk takes the remainder) front-loads the copies so the un-overlapped tail --
     * the last chunk's kernel and D2H -- is short */
    const bool pairs = f64 == 2; /* proba points at {float proba; int32 label} records, label is ignored */
    const bool full = f64 == 3;  /* proba points at b2f_scored_full records */
    if (full && !m->outlier) return set_err(B2F_ESTATE, "no outlier forest attached (b2f_model_attach_outlier_forest)");
    if (full && fmt == B2F_ROWS_RANKED)
        return set_err(B2F_EINVAL, "b2f_predict_full takes float32 rows (B2F_ROWS_WORDS24 / B2F_ROWS_PACKED64): ranks are relative to ONE forest's split values");
    if ((pairs || full) && !proba) return set_err(B2F_EINVAL, "out is NULL");
    int c = 0;
    for (int64_t off = 0; off < n; ++c) {
        int64_t cnt = std::min(chunk, n - off);
        if (!m->chunk_plan.empty() && chunk != n && n >= 2 * m->chunk_rows) {
            cnt = (size_t)c < m->chunk_plan.size() ? std::max<int64_t>(1024, (n * m->chunk_plan[c] / 1024 + 1023) / 1024 * 1024) : n - off;
            cnt = std::min(cnt, n - off);
        }
        struct Advance {
            int64_t &o, d;
            ~Advance() { o += d; }
        } advance{off, cnt};
        /* slots rotate ACROSS calls too, so with several batches in flight (async ring, stream dealer) the next
         * batch's H2D does not wait for the previous batch's kernel to release the same staging buffer */
        const int slot_idx = (int)((m->next_slot + (uint64_t)c) % B2F_STREAMS);
        Slot &sl = m->slots[slot_idx];
        int rc = slot_reserve(m, sl, cnt);
        if (rc) return rc;
        if (c == 0) mark(sl.stream);
        CUDA_TRY(cudaMemcpyAsync(sl.d_rows, static_cast<const uint8_t *>(rows) + (size_t)off * row_bytes, (size_t)cnt * row_bytes,
                                 cudaMemcpyHostToDevice, sl.stream));
        mark(sl.stream);
        if (full) { /* classifier, then the outlier forest, on the same device rows; 24-byte records, ONE D2H copy */
            static_assert(sizeof(b2f_scored_full) == 24 && offsetof(b2f_scored_full, label) == 8 && offsetof(b2f_scored_full, is_outlier) == 12 &&
                              offsetof(b2f_scored_full, outlier_score) == 16,
                          "b2f_scored_full layout");
            uint8_t *rec = static_cast<uint8_t *>(sl.d_proba);
            rc = launch_predict(m, sl.stream, sl.d_rows, cnt, fmt, rec, 1, reinterpret_cast<int32_t *>(rec + 8), B2F_OSTRIDE(3, 6));
            if (rc) return rc;
            rc = launch_predict(m->outlier, sl.stream, sl.d_rows, cnt, fmt, rec + 16, 0, reinterpret_cast<int32_t *>(rec + 12), B2F_OSTRIDE(6, 6));
            if (rc) return rc;
            mark(sl.stream);
            CUDA_TRY(cudaMemcpyAsync(static_cast<uint8_t *>(proba) + (size_t)off * sizeof(b2f_scored_full), sl.d_proba,
                                     (size_t)cnt * sizeof(b2f_scored_full), cudaMemcpyDeviceToHost, sl.stream));
            mark(sl.stream);
            *used_mask |= 1u << slot_idx;
            continue;
        }
        if (pairs) { /* one interleaved device buffer, ONE D2H copy per chunk */
            rc = launch_predict(m, sl.stream, sl.d_rows, cnt, fmt, sl.d_proba, 0, static_cast<int32_t *>(sl.d_proba) + 1, 2);
            if (rc) return rc;
            mark(sl.stream);
            CUDA_TRY(cudaMemcpyAsync(static_cast<uint8_t *>(proba) + (size_t)off * 8, sl.d_proba, (size_t)cnt * 8, cudaMemcpyDeviceToHost, sl.stream));
            mark(sl.stream);
            *used_mask |= 1u << slot_idx;
            continue;
        }
        rc = launch_predict(m, sl.stream, sl.d_rows, cnt, fmt, proba ? sl.d_proba : nullptr, f64, label ? sl.d_label : nullptr);
        if (rc) return rc;
        mark(sl.stream);
        if (proba)
            CUDA_TRY(cudaMemcpyAsync(static_cast<uint8_t *>(proba) + (size_t)off * psz, sl.d_proba, (size_t)cnt * psz, cudaMemcpyDeviceToHost, sl.stream));
        if (label) CUDA_TRY(cudaMemcpyAsync(label + off, sl.d_label, (size_t)cnt * sizeof(int32_t), cudaMemcpyDeviceToHost, sl.stream));
        mark(sl.stream);
        *used_mask |= 1u << slot_idx;
    }
    m->next_slot += (uint64_t)c;
    if (timeline) {
        cudaDeviceSynchronize();
        fprintf(stderr, "[b2f timeline] n=%lld chunk=%lld :", (long long)n, (long long)chunk);
        for (size_t i = 1; i < tev.size(); ++i) {
            float ms = 0;
            cudaEventElapsedTime(&ms, tev[0], tev[i]);
            fprintf(stderr, " %s%.1f", (i % 3 == 1) ? "| h2d " : (i % 3 == 2 ? "k " : "d2h "), ms * 1e3f);
        }
        fprintf(stderr, " (us)\n");
        for (auto e : tev) cudaEventDestroy(e);
    }
    return B2F_OK;
}

static int sync_mask(b2f_model *m, uint32_t mask) {
    for (int s = 0; s < B2F_STREAMS; ++s)
        if (mask & (1u << s)) CUDA_TRY(cudaStreamSynchronize(m->slots[s].stream));
    return B2F_OK;
}

static int predict_host(b2f_model *m, const void *rows, int64_t n, int fmt, void *proba, int f64, int32_t *label) {
    if (!m) return set_err(B2F_EINVAL, "model is NULL");
    uint32_t mask = 0;
    int rc = enqueue_host_batch(m, rows, n, fmt, proba, f64, label, &mask);
    int rc2 = sync_mask(m, mask);
    return rc ? rc : rc2;
}

extern "C" int b2f_predict(b2f_model *m, const void *rows, int64_t n, float *proba1, int32_t *label) {
    return predict_host(m, rows, n, B2F_ROWS_WORDS24, proba1, 0, label);
}
extern "C" int b2f_predict_f64(b2f_model *m, const void *rows, int64_t n, double *proba1, int32_t *label) {
    return predict_host(m, rows, n, B2F_ROWS_WORDS24, proba1, 1, label);
}
extern "C" int b2f_predict_ex(b2f_model *m, const void *rows, int64_t n, int row_format, void *proba1, int proba_is_f64, int32_t *label) {
    return predict_host(m, rows, n, row_format, proba1, proba_is_f64 ? 1 : 0, label);
}
extern "C" int b2f_predict_pairs(b2f_model *m, const void *rows, int64_t n, int row_format, b2f_scored *out) {
    if (!out && n > 0) return set_err(B2F_EINVAL, "out is NULL");
    return predict_host(m, rows, n, row_format, out, 2, nullptr);
}

extern "C" int b2f_model_attach_outlier_forest(b2f_model *m, const void *forest_blob, size_t nbytes) {
    if (!m) return set_err(B2F_EINVAL, "model is NULL");
    b2f_blob_header h;
    int rc = validate_blob(static_cast<const uint8_t *>(forest_blob), nbytes, &h);
    if (rc) return rc;
    if (h.agg_mode != B2F_AGG_IFOREST) return set_err(B2F_EINVAL, "outlier forest: agg_mode %u is not B2F_AGG_IFOREST", h.agg_mode);
    if (h.n_cat != m->hdr.n_cat || h.n_num != m->hdr.n_num)
        return set_err(B2F_EINVAL, "outlier forest: row schema (%u categorical, %u numeric) differs from the model's (%u, %u)", h.n_cat, h.n_num,
                       m->hdr.n_cat, m->hdr.n_num);
    b2f_model *child = b2f_model_create(forest_blob, nbytes, m->device);
    if (!child) return B2F_ECUDA; /* message set by b2f_model_create */
    CUDA_TRY(cudaSetDevice(m->device));
    if (m->outlier) {
        CUDA_TRY(cudaDeviceSynchronize());
        b2f_model_destroy(m->outlier);
    }
    m->outlier = child;
    return B2F_OK;
}

extern "C" int b2f_predict_full(b2f_model *m, const void *rows, int64_t n, int row_format, b2f_scored_full *out) {
    return predict_host(m, rows, n, row_format, out, 3, nullptr);
}

extern "C" int b2f_predict_async(b2f_model *m, const void *rows_pinned, int64_t n, void *proba1_pinned, int proba_is_f64,
                                 int32_t *label_pinned, b2f_ticket *ticket) {
    return b2f_predict_async_ex(m, rows_pinned, n, B2F_ROWS_WORDS24, proba1_pinned, proba_is_f64, label_pinned, ticket);
}

extern "C" int b2f_predict_async_ex(b2f_model *m, const void *rows_pinned, int64_t n, int row_format, void *proba1_pinned, int proba_is_f64,
                                    int32_t *label_pinned, b2f_ticket *ticket) {
    if (!m || !ticket) return set_err(B2F_EINVAL, "null argument");
    if (proba_is_f64 < 0 || proba_is_f64 > 3) return set_err(B2F_EINVAL, "proba_is_f64 = %d: expected 0 (float), 1 (double), 2 (b2f_scored) or 3 (b2f_scored_full)", proba_is_f64);
    if (proba_is_f64 >= 2 && n > 0 && !proba1_pinned) return set_err(B2F_EINVAL, "record output requested but the output pointer is NULL");
    const uint64_t id = m->next_ticket++;
    TicketRec &t = m->tickets[id % B2F_TICKETS];
    if (t.id != 0) { /* oldest ticket still outstanding in this ring position: retire it */
        for (int s = 0; s < B2F_STREAMS; ++s)
            if (t.used_mask & (1u << s)) CUDA_TRY(cudaEventSynchronize(t.ev[s]));
    }
    uint32_t mask = 0;
    int rc = enqueue_host_batch(m, rows_pinned, n, row_format, proba1_pinned, proba_is_f64, label_pinned, &mask);
    if (rc) {
        sync_mask(m, mask);
        return rc;
    }
    for (int s = 0; s < B2F_STREAMS; ++s)
        if (mask & (1u << s)) {
            if (!t.ev[s]) CUDA_TRY(cudaEventCreateWithFlags(&t.ev[s], cudaEventDisableTiming));
            CUDA_TRY(cudaEventRecord(t.ev[s], m->slots[s].stream));
        }
    t.id = id;
    t.used_mask = mask;
    *ticket = id;
    return B2F_OK;
}

extern "C" int b2f_wait(b2f_model *m, b2f_ticket ticket) {
    if (!m) return set_err(B2F_EINVAL, "model is NULL");
    TicketRec &t = m->tickets[ticket % B2F_TICKETS];
    if (t.id != ticket) return B2F_OK; /* already retired */
    CUDA_TRY(cudaSetDevice(m->device));
    for (int s = 0; s < B2F_STREAMS; ++s)
        if (t.used_mask & (1u << s)) CUDA_TRY(cudaEventSynchronize(t.ev[s]));
    t.id = 0;
    t.used_mask = 0;
    return B2F_OK;
}

extern "C" int b2f_predict_multi(b2f_model **models, int n_models, const void *rows, int64_t n, void *proba1, int proba_is_f64, int32_t *label) {
    return b2f_predict_multi_ex(models, n_models, rows, n, B2F_ROWS_WORDS24, proba1, proba_is_f64, label);
}

extern "C" int b2f_predict_multi_ex(b2f_model **models, int n_models, const void *rows, int64_t n, int row_format, void *proba1, int proba_is_f64,
                                    int32_t *label) {
    if (!models || n_models <= 0) return set_err(B2F_EINVAL, "no models");
    const size_t row_bytes = row_bytes_of(models[0], row_format);
    if (n < 0) return set_err(B2F_EINVAL, "negative row count");
    std::vector<uint32_t> masks(n_models, 0);
    /* 0 = float, 1 = double, 2 = b2f_scored records, 3 = b2f_scored_full records */
    const size_t psz = proba_is_f64 == 3 ? sizeof(b2f_scored_full) : (proba_is_f64 ? sizeof(double) : sizeof(float));
    int rc = B2F_OK;
    for (int i = 0; i < n_models && rc == B2F_OK; ++i) {
        const int64_t lo = n * i / n_models, hi = n * (i + 1) / n_models;
        if (hi <= lo) continue;
        rc = enqueue_host_batch(models[i], static_cast<const uint8_t *>(rows) + (size_t)lo * row_bytes, hi - lo, row_format,
                                proba1 ? static_cast<uint8_t *>(proba1) + (size_t)lo * psz : nullptr, proba_is_f64, label ? label + lo : nullptr,
                                &masks[i]);
    }
    for (int i = 0; i < n_models; ++i) {
        cudaSetDevice(models[i]->device);
        int rc2 = sync_mask(models[i], masks[i]);
        if (rc == B2F_OK) rc = rc2;
    }
    return rc;
}

static void bind_thread_near(int device); /* scorer.h */

/* Round-robin streaming over the GPUs of one box: batch b (rows [b*batch, (b+1)*batch)) goes to model b % n_models.
 * One host thread per GPU submits that GPU's batches through the asynchronous ring (at most `inflight` batches in
 * flight per GPU), so submission cost is paid in parallel; rows are independent, so there is no inter-GPU traffic. */
extern "C" int b2f_predict_stream(b2f_model **models, int n_models, const void *rows, int64_t n, int64_t batch, int row_format, void *proba1,
                                  int proba_is_f64, int32_t *label, int inflight) {
    if (!models || n_models <= 0 || batch <= 0 || n < 0) return set_err(B2F_EINVAL, "bad argument");
    if (inflight < 1) inflight = 1;
    if (inflight > 8) inflight = 8;
    const size_t row_bytes = row_bytes_of(models[0], row_format);
    const size_t psz = proba_is_f64 ? sizeof(double) : sizeof(float);
    const int64_t n_batches = (n + batch - 1) / batch;
    std::vector<int> rcs(n_models, B2F_OK);
    std::vector<std::string> msgs(n_models);
    auto worker = [&](int d) {
        b2f_model *m = models[d];
        bind_thread_near(m->device); /* submit from the GPU's own NUMA node (scorer.h) */
        std::vector<b2f_ticket> ring;
        int rc = B2F_OK;
        for (int64_t b = d; b < n_batches && rc == B2F_OK; b += n_models) {
            const int64_t lo = b * batch, cnt = std::min(batch, n - lo);
            if ((int)ring.size() >= inflight) {
                rc = b2f_wait(m, ring.front());
                ring.erase(ring.begin());
                if (rc) break;
            }
            b2f_ticket t = 0;
            rc = b2f_predict_async_ex(m, static_cast<const uint8_t *>(rows) + (size_t)lo * row_bytes, cnt, row_format,
                                      proba1 ? static_cast<uint8_t *>(proba1) + (size_t)lo * psz : nullptr, proba_is_f64, label ? label + lo : nullptr, &t);
            if (rc == B2F_OK) ring.push_back(t);
        }
        for (b2f_ticket t : ring) {
            int rc2 = b2f_wait(m, t);
            if (rc == B2F_OK) rc = rc2;
        }
        rcs[d] = rc;
        if (rc) msgs[d] = b2f_last_error(); /* the message is thread-local: carry it back */
    };
    std::vector<std::thread> threads;
    for (int d = 0; d < n_models; ++d) threads.emplace_back(worker, d); /* every GPU its own thread: the caller's affinity is left alone */
    for (auto &t : threads) t.join();
    for (int d = 0; d < n_models; ++d)
        if (rcs[d]) return set_err(rcs[d], "GPU %d: %s", models[d]->device, msgs[d].c_str());
    return B2F_OK;
}

/* ------------------------------------------------------------------ device-resident interface */
extern "C" void *b2f_device_alloc(b2f_model *m, size_t nbytes) {
    if (!m) return nullptr;
    void *p = nullptr;
    if (cudaSetDevice(m->device) != cudaSuccess || cudaMalloc(&p, nbytes ? nbytes : 1) != cudaSuccess) {
        set_err(B2F_ENOMEM, "cudaMalloc(%zu) failed: %s", nbytes, cudaGetErrorString(cudaGetLastError()));
        return nullptr;
    }
    return p;
}
extern "C" void b2f_device_free(b2f_model *m, void *dptr) {
    if (!m || !dptr) return;
    cudaSetDevice(m->device);
    cudaFree(dptr);
}
extern "C" int b2f_copy_h2d(b2f_model *m, void *dst_dev, const void *src_host, size_t nbytes) {
    if (!m) return set_err(B2F_EINVAL, "model is NULL");
    CUDA_TRY(cudaSetDevice(m->device));
    CUDA_TRY(cudaMemcpyAsync(dst_dev, src_host, nbytes, cudaMemcpyHostToDevice, m->compute));
    CUDA_TRY(cudaStreamSynchronize(m->compute));
    return B2F_OK;
}
extern "C" int b2f_copy_d2h(b2f_model *m, void *dst_host, const void *src_dev, size_t nbytes) {
    if (!m) return set_err(B2F_EINVAL, "model is NULL");
    CUDA_TRY(cudaSetDevice(m->device));
    CUDA_TRY(cudaMemcpyAsync(dst_host, src_dev, nbytes, cudaMemcpyDeviceToHost, m->compute));
    CUDA_TRY(cudaStreamSynchronize(m->compute));
    return B2F_OK;
}
extern "C" int b2f_predict_device(b2f_model *m, const void *rows_dev, int64_t n, void *proba1_dev, int proba_is_f64, int32_t *label_dev) {
    return b2f_predict_device_ex(m, rows_dev, n, B2F_ROWS_WORDS24, proba1_dev, proba_is_f64, label_dev);
}
extern "C" int b2f_predict_device_ex(b2f_model *m, const void *rows_dev, int64_t n, int row_format, void *proba1_dev, int proba_is_f64,
                                     int32_t *label_dev) {
    if (!m) return set_err(B2F_EINVAL, "model is NULL");
    int rcf = check_row_format(m, row_format);
    if (rcf) return rcf;
    CUDA_TRY(cudaSetDevice(m->device));
    return launch_predict(m, m->compute, rows_dev, n, row_format, proba1_dev, proba_is_f64, label_dev);
}
extern "C" int b2f_sync(b2f_model *m) {
    if (!m) return set_err(B2F_EINVAL, "model is NULL");
    CUDA_TRY(cudaSetDevice(m->device));
    CUDA_TRY(cudaStreamSynchronize(m->compute));
    return B2F_OK;
}

static int ensure_flush(b2f_model *m) {
    if (!m->d_flush) CUDA_TRY(cudaMalloc(&m->d_flush, B2F_FLUSH_BYTES));
    return B2F_OK;
}

extern "C" int b2f_predict_device_timed(b2f_model *m, const void *rows_dev, int64_t n, void *proba1_dev, int proba_is_f64, int32_t *label_dev,
                                        int iters, int flush_l2, float *ms_each) {
    if (!m || iters <= 0 || !ms_each) return set_err(B2F_EINVAL, "bad argument");
    CUDA_TRY(cudaSetDevice(m->device));
    if (flush_l2) {
        int rc = ensure_flush(m);
        if (rc) return rc;
    }
    std::vector<cudaEvent_t> ev(2 * (size_t)iters);
    for (auto &e : ev) CUDA_TRY(cudaEventCreate(&e));
    int rc = B2F_OK;
    for (int i = 0; i < iters && rc == B2F_OK; ++i) {
        if (flush_l2) CUDA_TRY(cudaMemsetAsync(m->d_flush, i & 0xff, B2F_FLUSH_BYTES, m->compute));
        CUDA_TRY(cudaEventRecord(ev[2 * i], m->compute));
        rc = launch_predict(m, m->compute, rows_dev, n, B2F_ROWS_WORDS24, proba1_dev, proba_is_f64, label_dev);
        CUDA_TRY(cudaEventRecord(ev[2 * i + 1], m->compute));
    }
    CUDA_TRY(cudaStreamSynchronize(m->compute));
    for (int i = 0; i < iters; ++i) CUDA_TRY(cudaEventElapsedTime(&ms_each[i], ev[2 * i], ev[2 * i + 1]));
    for (auto &e : ev) cudaEventDestroy(e);
    return rc;
}

/* Streaming measurement: `steps` launches over a pool of `pool` distinct device-resident batches
 * (batch i%pool), so consecutive steps read different HBM lines (pool * n * 96 B should exceed L2).
 * Per-launch events and one region event pair, all on the launching stream. */
extern "C" int b2f_predict_stream_timed(b2f_model *m, const void *rows_dev, int64_t n, int pool, void *proba1_dev, int proba_is_f64,
                                        int32_t *label_dev, int steps, float *ms_each, float *ms_total) {
    return b2f_predict_stream_timed_ex(m, rows_dev, n, B2F_ROWS_WORDS24, pool, proba1_dev, proba_is_f64, label_dev, steps, ms_each, ms_total);
}

extern "C" int b2f_predict_stream_timed_ex(b2f_model *m, const void *rows_dev, int64_t n, int row_format, int pool, void *proba1_dev,
                                           int proba_is_f64, int32_t *label_dev, int steps, float *ms_each, float *ms_total) {
    if (!m || steps <= 0 || pool <= 0 || !ms_total) return set_err(B2F_EINVAL, "bad argument");
    {
        int rcf = check_row_format(m, row_format);
        if (rcf) return rcf;
    }
    const size_t row_bytes = row_bytes_of(m, row_format);
    CUDA_TRY(cudaSetDevice(m->device));
    /* per-launch events only when the caller asks for per-launch times: an event record between two launches keeps
     * them from overlapping (programmatic dependent launch of the rank kernel), so the region time is measured without */
    const bool each = ms_each != nullptr;
    std::vector<cudaEvent_t> ev(each ? 2 * (size_t)steps + 2 : 2);
    for (auto &e : ev) CUDA_TRY(cudaEventCreate(&e));
    const size_t psz = proba_is_f64 ? sizeof(double) : sizeof(float);
    const size_t i0 = ev.size() - 2, i1 = ev.size() - 1;
    int rc = B2F_OK;
    CUDA_TRY(cudaEventRecord(ev[i0], m->compute));
    for (int i = 0; i < steps && rc == B2F_OK; ++i) {
        const size_t b = (size_t)(i % pool);
        if (each) CUDA_TRY(cudaEventRecord(ev[2 * i], m->compute));
        rc = launch_predict(m, m->compute, static_cast<const uint8_t *>(rows_dev) + b * (size_t)n * row_bytes, n, row_format,
                            proba1_dev ? static_cast<uint8_t *>(proba1_dev) + b * (size_t)n * psz : nullptr, proba_is_f64,
                            label_dev ? label_dev + b * (size_t)n : nullptr);
        if (each) CUDA_TRY(cudaEventRecord(ev[2 * i + 1], m->compute));
    }
    CUDA_TRY(cudaEventRecord(ev[i1], m->compute));
    CUDA_TRY(cudaStreamSynchronize(m->compute));
    if (each)
        for (int i = 0; i < steps; ++i) CUDA_TRY(cudaEventElapsedTime(&ms_each[i], ev[2 * i], ev[2 * i + 1]));
    CUDA_TRY(cudaEventElapsedTime(ms_total, ev[i0], ev[i1]));
    for (auto &e : ev) cudaEventDestroy(e);
    return rc;
}

/* ------------------------------------------------------------------ moments */
static int launch_moments(b2f_model *m, const void *rows_dev, int64_t n) {
    /* one CTA per 256-row slab up to a full wave of 3 CTAs per SM; small inputs get fewer CTAs so the
     * fixed-order final reduction over block partials stays short */
    const int64_t n_slabs = (n + B2F_MOM_SLAB_ROWS - 1) / B2F_MOM_SLAB_ROWS;
    int64_t blocks = std::min<int64_t>(m->mom_blocks, std::max<int64_t>(std::min<int64_t>(n_slabs, m->sm_count), n_slabs / 4));
    if (blocks < 1) blocks = 1;
    k_feature_moments<<<(unsigned)blocks, B2F_MOM_THREADS, B2F_MOM_SMEM, m->compute>>>(static_cast<const uint4 *>(rows_dev), (long long)n,
                                                                                     (int)m->hdr.n_cat, m->d_mom_partials, m->d_mom_ticket, m->d_mom_out);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return set_err(B2F_ECUDA, "k_feature_moments launch failed: %s", cudaGetErrorString(e));
    m->launches++;
    return B2F_OK;
}

extern "C" int b2f_moments_device(b2f_model *m, const void *rows_dev, int64_t n, double *out) {
    if (!m || !out || n < 0) return set_err(B2F_EINVAL, "bad argument");
    CUDA_TRY(cudaSetDevice(m->device));
    int rc = launch_moments(m, rows_dev, n);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(out, m->d_mom_out, B2F_MOM_VALUES * sizeof(double), cudaMemcpyDeviceToHost, m->compute));
    CUDA_TRY(cudaStreamSynchronize(m->compute));
    return B2F_OK;
}

static int moments_stage(b2f_model *m, const void *rows, int64_t n) {
    if (n > m->mom_cap_rows) {
        CUDA_TRY(cudaStreamSynchronize(m->compute));
        if (m->d_mom_rows) cudaFree(m->d_mom_rows);
        m->d_mom_rows = nullptr;
        m->mom_cap_rows = 0;
        CUDA_TRY(cudaMalloc(&m->d_mom_rows, (size_t)std::max<int64_t>(n, 1024) * B2F_ROW_BYTES));
        m->mom_cap_rows = std::max<int64_t>(n, 1024);
    }
    if (n > 0) CUDA_TRY(cudaMemcpyAsync(m->d_mom_rows, rows, (size_t)n * B2F_ROW_BYTES, cudaMemcpyHostToDevice, m->compute));
    return B2F_OK;
}

extern "C" int b2f_moments(b2f_model *m, const void *rows, int64_t n, double *out) {
    if (!m || !out || n < 0 || (n > 0 && !rows)) return set_err(B2F_EINVAL, "bad argument");
    CUDA_TRY(cudaSetDevice(m->device));
    int rc = moments_stage(m, rows, n);
    if (rc) return rc;
    return b2f_moments_device(m, m->d_mom_rows, n, out);
}

extern "C" int b2f_moments_device_timed(b2f_model *m, const void *rows_dev, int64_t n, int iters, int flush_l2, float *ms_each, double *out) {
    if (!m || iters <= 0 || !ms_each) return set_err(B2F_EINVAL, "bad argument");
    CUDA_TRY(cudaSetDevice(m->device));
    if (flush_l2) {
        int rc = ensure_flush(m);
        if (rc) return rc;
    }
    std::vector<cudaEvent_t> ev(2 * (size_t)iters);
    for (auto &e : ev) CUDA_TRY(cudaEventCreate(&e));
    int rc = B2F_OK;
    for (int i = 0; i < iters && rc == B2F_OK; ++i) {
        if (flush_l2) CUDA_TRY(cudaMemsetAsync(m->d_flush, i & 0xff, B2F_FLUSH_BYTES, m->compute));
        CUDA_TRY(cudaEventRecord(ev[2 * i], m->compute));
        rc = launch_moments(m, rows_dev, n);
        CUDA_TRY(cudaEventRecord(ev[2 * i + 1], m->compute));
    }
    if (out) CUDA_TRY(cudaMemcpyAsync(out, m->d_mom_out, B2F_MOM_VALUES * sizeof(double), cudaMemcpyDeviceToHost, m->compute));
    CUDA_TRY(cudaStreamSynchronize(m->compute));
    for (int i = 0; i < iters; ++i) CUDA_TRY(cudaEventElapsedTime(&ms_each[i], ev[2 * i], ev[2 * i + 1]));
    for (auto &e : ev) cudaEventDestroy(e);
    return rc;
}

/* Chan et al. pairwise merge of (count, mean, M2), in part order */
extern "C" void b2f_moments_merge(const double *parts, int k, double *out) {
    for (int w = 0; w < B2F_ROW_WORDS; ++w) {
        double n = 0.0, mean = 0.0, m2 = 0.0;
        for (int i = 0; i < k; ++i) {
            const double nb = parts[(size_t)i * B2F_MOM_VALUES + w * 3 + 0];
            const double mb = parts[(size_t)i * B2F_MOM_VALUES + w * 3 + 1];
            const double sb = parts[(size_t)i * B2F_MOM_VALUES + w * 3 + 2];
            if (nb <= 0.0) continue;
            if (n == 0.0) {
                n = nb, mean = mb, m2 = sb;
                continue;
            }
            const double tot = n + nb, delta = mb - mean;
            mean += delta * (nb / tot);
            m2 += sb + delta * delta * (n * nb / tot);
            n = tot;
        }
        out[w * 3 + 0] = n;
        out[w * 3 + 1] = mean;
        out[w * 3 + 2] = m2;
    }
}

/* ------------------------------------------------------------------ NCCL plumbing */
extern "C" int b2f_comm_unique_id(void *id_out128) {
    if (!id_out128) return set_err(B2F_EINVAL, "null argument");
    int rc = nccl_load();
    if (rc) return rc;
    ncclUniqueId id;
    NCCL_TRY(g_nccl.GetUniqueId(&id));
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    memcpy(id_out128, &id, 128);
    return B2F_OK;
}

static int comm_buffers(b2f_model *m, int nranks) {
    if (nranks > m->gather_cap) {
        if (m->d_gather) cudaFree(m->d_gather);
        m->d_gather = nullptr;
        CUDA_TRY(cudaMalloc(&m->d_gather, (size_t)(nranks + 1) * B2F_MOM_VALUES * sizeof(double)));
        m->gather_cap = nranks;
    }
    return B2F_OK;
}

extern "C" int b2f_comm_init_rank(b2f_model *m, int nranks, int rank, const void *id128) {
    if (!m || !id128 || nranks <= 0 || rank < 0 || rank >= nranks) return set_err(B2F_EINVAL, "bad argument");
    int rc = nccl_load();
    if (rc) return rc;
    CUDA_TRY(cudaSetDevice(m->device));
    ncclUniqueId id;
    memcpy(&id, id128, 128);
    NCCL_TRY(g_nccl.CommInitRank(&m->comm, nranks, id, rank));
    m->nranks = nranks;
    m->rank = rank;
    return comm_buffers(m, nranks);
}

extern "C" int b2f_comm_init_all(b2f_model **models, int n_models) {
    if (!models || n_models <= 0) return set_err(B2F_EINVAL, "no models");
    int rc = nccl_load();
    if (rc) return rc;
    std::vector<ncclComm_t> comms(n_models);
    std::vector<int> devs(n_models);
    for (int i = 0; i < n_models; ++i) devs[i] = models[i]->device;
    NCCL_TRY(g_nccl.CommInitAll(comms.data(), n_models, devs.data()));
    for (int i = 0; i < n_models; ++i) {
        models[i]->comm = comms[i];
        models[i]->nranks = n_models;
        models[i]->rank = i;
        CUDA_TRY(cudaSetDevice(models[i]->device));
        rc = comm_buffers(models[i], n_models);
        if (rc) return rc;
    }
    return B2F_OK;
}

extern "C" int b2f_moments_allgather(b2f_model *m, const double *local, double *merged) {
    if (!m || !local || !merged) return set_err(B2F_EINVAL, "null argument");
    if (!m->comm) return set_err(B2F_ESTATE, "communicator not initialised (call b2f_comm_init_rank)");
    CUDA_TRY(cudaSetDevice(m->device));
    double *send = m->d_gather + (size_t)m->nranks * B2F_MOM_VALUES;
    CUDA_TRY(cudaMemcpyAsync(send, local, B2F_MOM_VALUES * sizeof(double), cudaMemcpyHostToDevice, m->compute));
    NCCL_TRY(g_nccl.AllGather(send, m->d_gather, B2F_MOM_VALUES, ncclDouble, m->comm, m->compute));
    std::vector<double> parts((size_t)m->nranks * B2F_MOM_VALUES);
    CUDA_TRY(cudaMemcpyAsync(parts.data(), m->d_gather, parts.size() * sizeof(double), cudaMemcpyDeviceToHost, m->compute));
    CUDA_TRY(cudaStreamSynchronize(m->compute));
    b2f_moments_merge(parts.data(), m->nranks, merged);
    return B2F_OK;
}

extern "C" int b2f_moments_multi(b2f_model **models, int n_models, const void *rows, int64_t n, double *out) {
    if (!models || n_models <= 0 || !out || n < 0) return set_err(B2F_EINVAL, "bad argument");
    /* 1. every device reduces its contiguous slice */
    int rc = B2F_OK;
    for (int i = 0; i < n_models && rc == B2F_OK; ++i) {
        b2f_model *m = models[i];
        const int64_t lo = n * i / n_models, hi = n * (i + 1) / n_models;
        CUDA_TRY(cudaSetDevice(m->device));
        rc = moments_stage(m, static_cast<const uint8_t *>(rows) + (size_t)lo * B2F_ROW_BYTES, hi - lo);
        if (rc == B2F_OK) rc = launch_moments(m, m->d_mom_rows, hi - lo);
    }
    if (rc) return rc;
    const bool use_nccl = models[0]->comm != nullptr && models[0]->nranks == n_models;
    std::vector<double> parts((size_t)n_models * B2F_MOM_VALUES);
    if (use_nccl) {
        /* 2a. all-gather the 576-byte triples over NVLink; every rank ends up with all partials */
        NCCL_TRY(g_nccl.GroupStart());
        for (int i = 0; i < n_models; ++i) {
            b2f_model *m = models[i];
            ncclResult_t r = g_nccl.AllGather(m->d_mom_out, m->d_gather, B2F_MOM_VALUES, ncclDouble, m->comm, m->compute);
            if (r != ncclSuccess) {
                g_nccl.GroupEnd();
                return set_err(B2F_ENCCL, "ncclAllGather failed: %s", g_nccl.GetErrorString(r));
            }
        }
        NCCL_TRY(g_nccl.GroupEnd());
        CUDA_TRY(cudaSetDevice(models[0]->device));
        CUDA_TRY(cudaMemcpyAsync(parts.data(), models[0]->d_gather, parts.size() * sizeof(double), cudaMemcpyDeviceToHost, models[0]->compute));
        for (int i = 0; i < n_models; ++i) {
            CUDA_TRY(cudaSetDevice(models[i]->device));
            CUDA_TRY(cudaStreamSynchronize(models[i]->compute));
        }
    } else {
        /* 2b. no communicator: gather through the host */
        for (int i = 0; i < n_models; ++i) {
            CUDA_TRY(cudaSetDevice(models[i]->device));
            CUDA_TRY(cudaMemcpyAsync(parts.data() + (size_t)i * B2F_MOM_VALUES, models[i]->d_mom_out, B2F_MOM_VALUES * sizeof(double),
                                     cudaMemcpyDeviceToHost, models[i]->compute));
            CUDA_TRY(cudaStreamSynchronize(models[i]->compute));
        }
    }
    b2f_moments_merge(parts.data(), n_models, out);
    return B2F_OK;
}

/* ------------------------------------------------------------------ columnar request pipeline (encode -> H2D -> kernel -> D2H per chunk) */
#include "scorer.h"

/* ------------------------------------------------------------------ batch drift detector (K3) */
#include "drift_api.cuh"
