/*
 * forest_predict_rank.cuh -- K1c: the rank-quantised form of the fused scoring kernel (sm_100a), for forests that stay
 * resident in shared memory.  Same arithmetic as k_forest_predict / k_forest_predict_tile -- it replaces
 * `classifier.predict_proba(df[all_features])[:, 1]` (reference databricks/src/02-register-model.ipynb:335-337) -- on rows in
 * the B2F_ROWS_RANKED format (forest_rank.h): every numeric feature arrives as its rank among the forest's split values and
 * every tested (categorical feature, category) pair becomes a 0/1 value, so EVERY split is one unsigned integer compare
 * "value[f] >= t" and a node is ONE 32-bit word (t << 16 | byte offset of value[f] in the tile's value block).
 *
 * Why (round-1 ncu, profiles/r01_ncu_tile.txt): the walk is bound by shared-memory wavefronts (LSU pipe, 1 per clock per SM).
 * An 8-byte node costs two wavefronts per warp-level visit (LDS.64 is served half-warp by half-warp) plus a leaf-id load; here
 *   - a node is 4 bytes: one wavefront, and at most 32 consecutive words per level up to depth 5 -> never a bank conflict;
 *   - trees are COMPLETE in breadth-first order: child = 2i+1(+1), no child pointer, no leaf-id load -- after D levels the
 *     path bits ARE the leaf index;
 *   - per warp-level visit: LDS node, LOP3 (value address), LDS.U16 value, IMAD (value << 16 | 0xFFFF), ISETP, SEL, IMAD
 *     (child address): 3 ops on the integer ALU pipe, 2 on the FMA pipe.  (The first version tested categorical nodes by
 *     equality next to the numeric >=: 6 ALU-pipe ops per visit, and ncu showed that pipe -- one warp instruction per two
 *     cycles per scheduler -- at 77 %, i.e. the bound; profiles/r02_ncu_rank_v1.txt.)
 * and the machine is filled differently from the tile kernel (which left 60 % of its warps without a tile at 65 536 rows):
 *   - one CTA per SM, 32 warps, ALL of them walk; the CTA owns a contiguous run of 32-row tiles (<= 16 per round);
 *   - phase 1  all 1024 threads stage the CTA's rows into the per-tile value block xs[tile][f >> 1][lane][f & 1] (16-bit values,
 *              TRANSPOSED: lane l's values sit in bank l, so the per-lane dynamic fetch of the walk is one conflict-free
 *              LDS.U16), one lane per row and a share of the pseudo-features per thread, while one thread streams the forest
 *              into shared memory with TMA bulk copies (cp.async.bulk + mbarrier complete_tx);
 *   - phase 2  the round's work is tiles x tree groups (U trees per group, walked as U independent chains per thread; only the
 *              ceil(n_trees / U) groups that hold real trees); warp w takes the contiguous share [w * units / 32, (w+1) * units / 32)
 *              -- balanced to one tree group whatever the batch size -- and leaves one float64 partial per (warp, tile) it touched.
 *              The top two levels of a group come from its head record (RParams::head_off): 3U words that every lane needs, read
 *              as broadcast LDS.128, so a tree costs D - 2 per-lane node loads instead of D;
 *   - phase 3  one thread per row adds that row's partials in warp order (fixed order: deterministic), aggregates
 *              (RF mean | GBDT expit | isolation-forest score) and stores probability + label, coalesced.
 *   - STREAM = true (rank layouts larger than shared memory, e.g. 500 trees x depth 8 = 1.5 MB): the layout is cut into pieces of
 *     8 trees (2 tree groups) that travel through a two-slot ring -- thread 0 issues the TMA copy of piece k + 2 right after the
 *     barrier that ends piece k, so the copy overlaps the walk of piece k + 1 -- and warp w owns (tile w / 2, group w mod 2) of
 *     EVERY piece: its float64 sum stays in a register across the whole forest (<= 16 tiles per round).
 *   - launched with programmatic stream serialization (PDL): `griddepcontrol.launch_dependents` is issued at entry so the next
 *     launch's CTAs take over SMs as this launch's CTAs retire; `griddepcontrol.wait` sits before the first global STORE (phase 3),
 *     so forest fill, row staging and the walk all overlap the previous launch's tail.  Reading rows before the wait is safe
 *     because the host launches without PDL whenever the rows overlap the outputs of any rank launch still chained to this
 *     one through PDL on that stream (b2f_api.cu rank_launch_pdl), and no other kernel triggers its dependents early.
 */
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "forest_predict.cuh"
#include "forest_predict_tile.cuh"

#define B2F_RANK_THREADS 1024
#define B2F_RANK_WARPS 32
#define B2F_RANK_MAX_TILES 16                       /* 32-row tiles per CTA per round */
#define B2F_RANK_XS_BYTES 8192                      /* per tile: 64 words x 32 lanes x 4 B (128 16-bit values per lane), 8 KB aligned */
#define B2F_RANK_PARTIALS (B2F_RANK_WARPS + B2F_RANK_MAX_TILES)

struct RParams {
    const uint8_t *layout;   /* device: n_trees_padded complete trees, tree_stride bytes each; resident: then the head table */
    uint32_t layout_bytes;   /* multiple of 16 (resident: trees + head table) */
    uint32_t tree_stride;    /* 2^D * 12 */
    int32_t n_trees_padded;  /* multiple of 8 */
    int32_t n_groups;        /* resident: tree groups walked per tile = ceil(n_trees / U) (the stub trees past them add 0.0) */
    uint32_t head_off;       /* resident: byte offset of the head table, 3U words per group of U trees: the U root words, then
                                the U (left, right) level-1 word pairs (16-byte aligned, so a group's heads are 3U/4 LDS.128) */
    int32_t depth;
    int32_t agg_mode;
    int32_t n_cat;
    int32_t n_num;
    int32_t row_bytes;       /* multiple of 8 */
    int32_t cat_bytes;       /* 4 or 8 */
    int32_t max_tiles;       /* tiles per round (<= B2F_RANK_MAX_TILES, what shared memory allows) */
    int32_t n_pieces;        /* STREAM: pieces per pass over the forest; piece = groups_per_piece tree groups, piece_bytes bytes */
    int32_t groups_per_piece;
    uint32_t piece_bytes;
    double init_raw;
    double denom;
    double threshold;
    uint32_t mul_two;        /* = 2, mul_64k = 65536, add_64k = 65535: multiplier / addend operands handed over as run-time values so */
    uint32_t mul_64k;        /*   ptxas keeps the two multiply-adds of a node visit as IMAD (FMA pipe) instead of strength-reducing */
    uint32_t add_64k;        /*   them to LEA / IADD3 on the integer ALU pipe, which is the pipe that bounds the walk */
    int32_t n_pairs;         /* tested (categorical feature, category) pairs = pseudo-features even(n_num) .. + n_pairs - 1 */
    uint8_t cat_shift[16];   /* bit position / width of categorical field j inside the row's categorical block */
    uint8_t cat_bits[16];
    uint8_t cat_start[16];   /* pair index of feature j's first tested category (pairs are sorted by feature, then category) */
    unsigned long long cat_mask[16]; /* bit c set: category c of feature j is tested by some node */
#ifdef B2F_RANK_TRACE
    unsigned long long *trace; /* B2F_RANK_TRACE_WORDS words per CTA of this launch (see RANK_TRACE below) */
#endif
};

/* B2F_RANK_TRACE (off in the normal build; tools/rank_phases.py builds a traced copy): thread 0 of every CTA records its SM
 * and %globaltimer at the kernel's phase boundaries, so the time between launches can be split into phases */
#define B2F_RANK_TRACE_WORDS 8
#define B2F_RANK_TRACE_LAUNCHES 256
enum { RT_SMID, RT_ENTRY, RT_FOREST, RT_WAIT, RT_STAGED, RT_WALKED, RT_EXIT };
#ifdef B2F_RANK_TRACE
__device__ __forceinline__ unsigned long long rank_trace_now() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ unsigned long long rank_trace_smid() {
    uint32_t s;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(s));
    return s;
}
#define RANK_TRACE(i)                                                                                                       \
    do {                                                                                                                    \
        if (threadIdx.x == 0)                                                                                               \
            p.trace[(size_t)blockIdx.x * B2F_RANK_TRACE_WORDS + (i)] = (i) == RT_SMID ? rank_trace_smid() : rank_trace_now(); \
    } while (0)
#else
#define RANK_TRACE(i) \
    do {              \
    } while (0)
#endif

__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

__device__ __forceinline__ uint32_t lds_u16(uint32_t a) {
    uint32_t v;
    asm volatile("{ .reg .u16 h; ld.shared.u16 h, [%1]; cvt.u32.u16 %0, h; }" : "=r"(v) : "r"(a));
    return v;
}

/* levels D0 .. D-1 of U chains, then the payloads (added in tree order).  A chain keeps the ABSOLUTE shared address a = B + 4i of
 * its node (B = the tree's base): the child 2i+1 (+1) sits at 2a - B + 4 (+4), i.e. one SEL between the two per-tree constants
 * (k4 = 4 - B, k8 = 8 - B) and one multiply-add (FMA pipe). */
template <int D0, int D, int U>
__device__ __forceinline__ void rank_walk_levels(uint32_t (&at)[U], const uint32_t (&k4)[U], const uint32_t (&k8)[U], uint32_t xs_lane, uint32_t m2,
                                                 uint32_t m64k, uint32_t a64k, double &acc) {
#pragma unroll
    for (int d = D0; d < D; ++d) {
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint32_t nw = lds32(at[u]);
            const uint32_t v = lds_u16(xs_lane | (nw & 0x1F82u)); /* value[f] of this lane's row */
            const uint32_t x = v * m64k + a64k;                   /* (v << 16 | 0xFFFF) >= node  <=>  v >= t   (IMAD) */
            at[u] = at[u] * m2 + (x >= nw ? k8[u] : k4[u]);       /* IMAD */
        }
    }
    /* a = B + 4 (2^D - 1 + leaf): payload at B + 4 * 2^D + 8 * leaf = 2a - B - 4 * 2^D + 8 = (a + a + k4) + (4 - 4 * 2^D) */
#pragma unroll
    for (int u = 0; u < U; ++u) acc += lds_f64(at[u] + at[u] + k4[u] + 4u - (4u << D));
}

/* walk U consecutive trees (first tree at shared address t0) for this lane's row, every level from the tree body (streamed pieces) */
template <int D, int U>
__device__ __forceinline__ void rank_walk_group(uint32_t t0, uint32_t tree_stride, uint32_t xs_lane, uint32_t m2, uint32_t m64k, uint32_t a64k,
                                                double &acc) {
    uint32_t at[U], k4[U], k8[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
        at[u] = t0 + u * tree_stride;
        k4[u] = 4u - at[u];
        k8[u] = 8u - at[u];
    }
    rank_walk_levels<0, D, U>(at, k4, k8, xs_lane, m2, m64k, a64k, acc);
}

/* the same walk with the top two levels taken from the group's head record (shared address hd): its 3U words are the same for
 * every lane, so they arrive as 3U/4 broadcast LDS.128 instead of 2U per-lane node loads; the root test SELects the level-1 word */
template <int D, int U>
__device__ __forceinline__ void rank_walk_group_head(uint32_t t0, uint32_t hd, uint32_t tree_stride, uint32_t xs_lane, uint32_t m2, uint32_t m64k,
                                                     uint32_t a64k, double &acc) {
    static_assert(U % 4 == 0, "head records are read 4 words at a time");
    uint32_t hw[3 * U];
#pragma unroll
    for (int q = 0; q < 3 * U / 4; ++q)
        asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];"
                     : "=r"(hw[4 * q]), "=r"(hw[4 * q + 1]), "=r"(hw[4 * q + 2]), "=r"(hw[4 * q + 3])
                     : "r"(hd + 16u * q));
    uint32_t at[U], k4[U], k8[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
        at[u] = t0 + u * tree_stride;
        k4[u] = 4u - at[u];
        k8[u] = 8u - at[u];
        const uint32_t r = hw[u];
        const bool c0 = lds_u16(xs_lane | (r & 0x1F82u)) * m64k + a64k >= r;
        at[u] = at[u] * m2 + (c0 ? k8[u] : k4[u]); /* node 1 or 2 */
        if constexpr (D >= 2) {
            const uint32_t n1 = c0 ? hw[U + 2 * u + 1] : hw[U + 2 * u];
            const bool c1 = lds_u16(xs_lane | (n1 & 0x1F82u)) * m64k + a64k >= n1;
            at[u] = at[u] * m2 + (c1 ? k8[u] : k4[u]); /* node 3 .. 6 */
        }
    }
    rank_walk_levels<(D >= 2 ? 2 : 1), D, U>(at, k4, k8, xs_lane, m2, m64k, a64k, acc);
}

template <int D, int U, bool STREAM, typename OutT>
__global__ void __launch_bounds__(B2F_RANK_THREADS, 1)
    k_forest_predict_rank(const __grid_constant__ RParams p, const uint8_t *__restrict__ rows, long long n, OutT *__restrict__ proba,
                          int32_t *__restrict__ label, int ostride) {
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ __align__(8) uint64_t forest_bar[2]; /* resident: [0] = the whole layout; STREAM: one per ring slot */

    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;

    pdl_launch_dependents(); /* the next launch may start filling SMs as this one's CTAs retire */
    RANK_TRACE(RT_SMID);
    RANK_TRACE(RT_ENTRY);

    /* shared-memory plan: [xs: max_tiles x 8 KB value blocks, 8 KB aligned][partials][forest | two-slot piece ring] */
    const uint32_t pad = (B2F_RANK_XS_BYTES - (smem_addr(smem) & (B2F_RANK_XS_BYTES - 1u))) & (B2F_RANK_XS_BYTES - 1u);
    uint8_t *xs_all = smem + pad;
    double *partial = reinterpret_cast<double *>(xs_all + (size_t)p.max_tiles * B2F_RANK_XS_BYTES);
    uint8_t *forest = reinterpret_cast<uint8_t *>(partial + B2F_RANK_PARTIALS * 32);

    if (tid == 0) {
        mbar_init(&forest_bar[0], 1);
        mbar_init(&forest_bar[1], 1);
        fence_mbar_init();
        fence_proxy_async();
        if constexpr (!STREAM) {
            /* the forest is launch-invariant (never written by a kernel): safe to fetch before griddepcontrol.wait */
            mbar_arrive_expect_tx(&forest_bar[0], p.layout_bytes);
            for (uint32_t o = 0; o < p.layout_bytes; o += B2F_BULK_PIECE) {
                const uint32_t part = min(B2F_BULK_PIECE, p.layout_bytes - o);
                tma_bulk_g2s(forest + o, p.layout + o, part, &forest_bar[0]);
            }
        }
    }
    /* STREAM: piece k (counted over all rounds) lands in slot k mod 2; issued by thread 0 only */
    auto issue_piece = [&](uint32_t k) {
        const uint32_t slot = k & 1u, piece = k % (uint32_t)p.n_pieces;
        mbar_arrive_expect_tx(&forest_bar[slot], p.piece_bytes);
        tma_bulk_g2s(forest + slot * p.piece_bytes, p.layout + (size_t)piece * p.piece_bytes, p.piece_bytes, &forest_bar[slot]);
    };

    /* this CTA's run of tiles (32-bit arithmetic: n < 2^31 rows) */
    const uint32_t n_tiles = (uint32_t)((n + 31) >> 5);
    const uint32_t tq = n_tiles / gridDim.x, tr = n_tiles % gridDim.x;
    const uint32_t tile0 = blockIdx.x * tq + min(blockIdx.x, tr), cta_tiles = tq + (blockIdx.x < tr ? 1u : 0u);
    const uint32_t n_rounds = (cta_tiles + (uint32_t)p.max_tiles - 1u) / (uint32_t)p.max_tiles;
    const int groups = p.n_groups; /* tree groups per tile (resident) */
    const uint32_t forest_addr = smem_addr(forest);
    const uint32_t xs_addr = smem_addr(xs_all);
    const uint32_t head_addr = forest_addr + p.head_off;
    bool forest_ready = false;

    for (uint32_t round = 0; round < n_rounds; ++round) {
        const uint32_t rt0 = cta_tiles * round / n_rounds, rt1 = cta_tiles * (round + 1u) / n_rounds;
        const int T = (int)(rt1 - rt0);
        const long long row0 = (long long)(tile0 + rt0) * 32;
        const int n_rows = (int)min((long long)T * 32, n - row0);
        if (round > 0) __syncthreads(); /* xs / partials of the previous round are free */

        /* ---- phase 1: stage rows.  item = (part, row): consecutive lanes take consecutive rows, so every store of a warp goes
         *      to 32 different banks.  part 0 copies the numeric ranks (two uint16 per 32-bit word in the row and in the block
         *      alike); part 1 clears the row's one-hot words and sets the <= n_cat values whose category some node tests ---- */
        {
            const int items = T * 32 * 2;
            const int num_words = (p.n_num + 1) >> 1, hot_words = (p.n_pairs + 1) >> 1;
            for (int it = tid; it < items; it += B2F_RANK_THREADS) {
                const int part = it >= T * 32 ? 1 : 0, r = it - part * (T * 32);
                const uint32_t col = xs_addr + (uint32_t)(r >> 5) * B2F_RANK_XS_BYTES + (uint32_t)(r & 31) * 4u;
                const bool live = r < n_rows;
                const uint8_t *row = rows + (size_t)(row0 + (live ? r : 0)) * p.row_bytes;
                if (part == 0) {
                    const uint32_t *q = reinterpret_cast<const uint32_t *>(row + p.cat_bytes);
                    for (int w = 0; w < num_words; ++w) {
                        uint32_t v = live ? __ldg(q + w) : 0u;
                        if (2 * w + 1 >= p.n_num) v &= 0xFFFFu; /* odd feature count: the upper half is padding of the row */
                        asm volatile("st.shared.u32 [%0], %1;" ::"r"(col + (uint32_t)w * 128u), "r"(v) : "memory");
                    }
                } else {
                    const uint32_t hot = col + (uint32_t)num_words * 128u;
                    for (int w = 0; w < hot_words; ++w) asm volatile("st.shared.u32 [%0], %1;" ::"r"(hot + (uint32_t)w * 128u), "r"(0u) : "memory");
                    if (live) {
                        unsigned long long cw = __ldg(reinterpret_cast<const uint32_t *>(row));
                        if (p.cat_bytes == 8) cw |= (unsigned long long)__ldg(reinterpret_cast<const uint32_t *>(row) + 1) << 32;
                        for (int j = 0; j < p.n_cat; ++j) {
                            const uint32_t code1 = (uint32_t)(cw >> p.cat_shift[j]) & ((1u << p.cat_bits[j]) - 1u);
                            const unsigned long long m = p.cat_mask[j];
                            if (code1 != 0u && code1 <= 64u && ((m >> (code1 - 1u)) & 1ull)) {
                                const uint32_t slot = (uint32_t)p.cat_start[j] + (uint32_t)__popcll(m & ((1ull << (code1 - 1u)) - 1ull));
                                asm volatile("st.shared.u16 [%0], %1;" ::"r"(hot + (slot >> 1) * 128u + (slot & 1u) * 2u), "h"((uint16_t)1) : "memory");
                            }
                        }
                    }
                }
            }
        }
        if constexpr (STREAM) {
            /* the first two pieces of this pass: both ring slots are free (every warp is past the previous pass's last barrier) */
            if (tid == 0) {
                issue_piece(round * (uint32_t)p.n_pieces);
                if (p.n_pieces > 1) issue_piece(round * (uint32_t)p.n_pieces + 1u);
            }
        }
        __syncthreads();
        RANK_TRACE(RT_STAGED);
        if constexpr (!STREAM) {
            if (!forest_ready) {
                mbar_wait(&forest_bar[0], 0);
                forest_ready = true;
            }
            RANK_TRACE(RT_FOREST);
        }

        if constexpr (STREAM) {
            /* ---- phase 2 (streamed): warp w owns (tile w / GP, group w mod GP) of every piece; the sum stays in a register ---- */
            const int GP = p.groups_per_piece;
            const bool mine = warp < T * GP;
            const uint32_t xs_lane = xs_addr + (uint32_t)(warp / GP) * B2F_RANK_XS_BYTES + (uint32_t)lane * 4u;
            const uint32_t g_off = (uint32_t)(warp % GP) * U * p.tree_stride;
            double acc = 0.0;
            for (int piece = 0; piece < p.n_pieces; ++piece) {
                const uint32_t k = round * (uint32_t)p.n_pieces + (uint32_t)piece;
                mbar_wait(&forest_bar[k & 1u], (k >> 1) & 1u);
                if (mine) rank_walk_group<D, U>(forest_addr + (k & 1u) * p.piece_bytes + g_off, p.tree_stride, xs_lane, p.mul_two, p.mul_64k, p.add_64k, acc);
                __syncthreads(); /* every warp is done with this slot: refill it while the other slot is walked */
                if (tid == 0 && piece + 2 < p.n_pieces) issue_piece(k + 2u);
            }
            if (mine) partial[warp * 32 + lane] = acc;
            __syncthreads();
            RANK_TRACE(RT_WALKED);
            pdl_wait(); /* before the first global store: see phase 3 of the resident path */
            RANK_TRACE(RT_WAIT);
            for (int r = tid; r < n_rows; r += B2F_RANK_THREADS) {
                const int t = r >> 5, ln = r & 31;
                double s = p.agg_mode == B2F_AGG_GBDT_LOGISTIC ? p.init_raw : 0.0;
                for (int g = 0; g < GP; ++g) s += partial[(t * GP + g) * 32 + ln];
                double p1;
                int lab;
                aggregate(p.agg_mode, p.agg_mode == B2F_AGG_GBDT_LOGISTIC ? 0.0 : p.init_raw, p.denom, p.threshold, s, p1, lab);
                const long long row = row0 + r;
                if (proba) proba[row * ostride_p(ostride)] = (OutT)p1;
                if (label) label[row * ostride_l(ostride)] = lab;
            }
            continue;
        }

        /* ---- phase 2: walk.  units = T x groups, warp w takes [w * units / 32, (w + 1) * units / 32) ---- */
        {
            const int units = T * groups;
            int u = warp * units / B2F_RANK_WARPS; /* units <= 16 tiles x 128 groups: 32-bit */
            const int u_end = (warp + 1) * units / B2F_RANK_WARPS;
            while (u < u_end) {
                const int t = u / groups;
                const int g_end = min(groups, u_end - t * groups);
                const uint32_t xs_lane = xs_addr + (uint32_t)t * B2F_RANK_XS_BYTES + (uint32_t)lane * 4u;
                double acc = 0.0;
                for (int g = u - t * groups; g < g_end; ++g)
                    rank_walk_group_head<D, U>(forest_addr + (uint32_t)(g * U) * p.tree_stride, head_addr + (uint32_t)g * (12u * U), p.tree_stride,
                                               xs_lane, p.mul_two, p.mul_64k, p.add_64k, acc);
                partial[(warp + t) * 32 + lane] = acc; /* slot (warp + tile) is unique to this (warp, tile) segment */
                u = t * groups + g_end;
            }
        }
        __syncthreads();
        RANK_TRACE(RT_WALKED);
        /* the first global store: the previous launch in the stream may still read these outputs (its rows) or write them.
         * Rows and forest were read before this point, which is safe because the host never lets a launch with programmatic
         * serialization read rows that an earlier rank launch of its programmatic chain writes (rank_launch_pdl), and the rank
         * kernel is the only kernel that triggers its dependents early (griddepcontrol.launch_dependents) */
        pdl_wait();
        RANK_TRACE(RT_WAIT);

        /* ---- phase 3: one thread per row: partials in warp order -> aggregate -> store ---- */
        for (int r = tid; r < n_rows; r += B2F_RANK_THREADS) {
            const int t = r >> 5, ln = r & 31;
            const int units = T * groups;
            /* warps whose share meets tile t: first and last unit of the tile are t*groups and (t+1)*groups - 1 */
            const int w_first = (int)(((uint32_t)(t * groups + 1) * B2F_RANK_WARPS + (uint32_t)units - 1u) / (uint32_t)units) - 1;
            const int w_last = (int)(((uint32_t)((t + 1) * groups) * B2F_RANK_WARPS + (uint32_t)units - 1u) / (uint32_t)units) - 1;
            double s = p.agg_mode == B2F_AGG_GBDT_LOGISTIC ? p.init_raw : 0.0;
            for (int w = w_first; w <= w_last; ++w) /* warps whose share is empty (units < 32) wrote nothing */
                if ((w + 1) * units / B2F_RANK_WARPS > w * units / B2F_RANK_WARPS) s += partial[(w + t) * 32 + ln];
            double p1;
            int lab;
            aggregate(p.agg_mode, p.agg_mode == B2F_AGG_GBDT_LOGISTIC ? 0.0 : p.init_raw, p.denom, p.threshold, s, p1, lab);
            const long long row = row0 + r;
            if (proba) proba[row * ostride_p(ostride)] = (OutT)p1;
            if (label) label[row * ostride_l(ostride)] = lab;
        }
    }
    if constexpr (!STREAM) {
        if (!forest_ready) mbar_wait(&forest_bar[0], 0); /* never retire a CTA while a bulk copy into its shared memory is in flight */
    }
    RANK_TRACE(RT_EXIT);
}
