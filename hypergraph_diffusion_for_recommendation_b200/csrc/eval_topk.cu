// Full-ranking evaluation: user x item score contraction fused with training-item masking and a
// per-user top-K, sm_100a.
//
// Replaces GraphRecommender.test (base/graph_recommender.py:61-92 = base/main_recommender.py:64-100):
//   for user in test_set:  candidates = predict(user)            # torch.matmul(user_emb[u], item_emb.T).cpu()
//                          candidates[train items of user] = -10e8
//                          ids, scores = find_k_largest(max_N, candidates)      # util/algorithm.py:143-173
// i.e. one GEMV + a PCIe copy of n_items floats + a python mask loop + a numba insertion top-K per user.
//
// Pipeline (all on the caller's stream, no host synchronisation):
//   1. eval_pack_kernel      fp32 tables -> two bf16 terms (hi + lo, 16 significant bits) in the tcgen05 K-major no-swizzle core-matrix layout
//                            (8 rows x 16 B core matrices; an 8-row group is 1 KB), row norms for the
//                            error bound.  A tile is then ONE contiguous block: a single cp.async.bulk.
//   2. eval_scores_kernel    the dense step, run twice.  CTA = 256 test users x a range of 128-item tiles.
//                            warp 0: bulk-copy producer (6-stage mbarrier ring); warp 1: one thread issues
//                            tcgen05.mma kind::f16 (bf16 x bf16 -> fp32, M128 N128 K16, 4 per half) into a
//                            double-buffered TMEM accumulator (2 stages x 2 halves x 128 columns = 512);
//                            warps 2..17: epilogue, tcgen05.ld 32x32b (thread = user row x 64-column half), the user's training
//                            items poisoned to NaN by walking the train CSR row in step with the columns.
//        SAMPLE pass         over 1/4 of the item tiles: 32 running bucket maxima per (user, item segment).
//        eval_tau_kernel     K-th largest bucket maximum = a lower bound tau of the user's K-th best score.
//        FILTER pass         over all item tiles: scores >= tau - 2 eps are appended to the user's candidate
//                            list.  Scores never leave the SM; only ~(4 K + window) (score, id) pairs per user do.
//                            Long lists (64 < K <= 256): one pool of up to 8 K slots per user, filled through a
//                            per-user append counter, instead of one short list per (sub-range, column half, user).
//   3. eval_rescore_kernel   approximate K-th best among the candidates prunes the list, the survivors are
//                            re-scored exactly in fp32 in the canonical order (ascending-k fused multiply-add,
//                            oracle/hgr_oracle.c hgr_oracle_scores_f32), exact top-K: score descending, ties by
//                            ascending item id.  |bf16 score - fp32 score| <= eps(user) is a proven bound, so
//                            the candidate set is a superset of the true top-K: bit-identical to the oracle.
//                            Long lists: one block per user sorts its pool in shared memory instead.
//   4. eval_brute_kernel     exact SIMT fallback for users whose candidate list overflowed (and the whole
//                            job when D != 64 or K > 256): every score in fp32, K rounds of block arg-max.
//   5. eval_refquirk_kernel  optional: replays find_k_largest's re-visit of the first K candidates
//                            (SURVEY.md F9) so that Recall/NDCG strings match the reference bit for bit.
//                            One warp per user for K <= 64, one block per user for long lists.
#include <cuda_bf16.h>
#include <math_constants.h>
#include <string.h>
#include <limits.h>

#include "hgr_internal.cuh"

namespace hgr {

// ------------------------------------------------------------------------------------------ constants
constexpr int EV_D = 64;           // embedding width of the tensor path (one 128-byte bf16 row)
constexpr int EV_BM = 256;         // users per CTA: two 128-row accumulators
constexpr int EV_BN = 128;         // items per tile
constexpr int EV_STAGES = 4;       // item tiles in flight (192 KB of shared memory: one CTA per SM, so its
                                   // 512-column TMEM allocation never waits)
constexpr int EV_A_BYTES = EV_BM * EV_D * 2;        // 32 KB per bf16 term (hi, lo)
constexpr int EV_B_BYTES = EV_BN * EV_D * 2;        // 16 KB per bf16 term (hi, lo)
constexpr int EV_CSPLIT = 2;                        // epilogue warps per (128-row half, TMEM lane quadrant): column halves of a tile
constexpr int EV_EPI_WARPS = 8 * EV_CSPLIT;         // 4 per scheduler: the epilogue is latency-bound with fewer
constexpr int EV_THREADS = 64 + 32 * EV_EPI_WARPS;  // producer warp, MMA warp, 16 epilogue warps
constexpr int EV_TMEM_COLS = 512;
constexpr int EV_SAMPLE_STRIDE = 4;                 // the sample pass scores 1 / 4 of the item tiles
constexpr int EV_BUCKETS = 32;                      // bucket maxima per (user, sample segment)
constexpr float EV_MASK_SCORE = -10e8f;             // base/graph_recommender.py:80
constexpr int EV_LIST_K = 64;                       // largest K of the per-(sub-range, column half, user) candidate lists
constexpr int EV_MAX_K = 256;                       // largest K of the tensor path: "long lists" are EV_LIST_K < K <= EV_MAX_K
constexpr int EV_POOL_PER_K = 8;                    // long lists: candidate slots per user, in multiples of K
// Every fp32 value x is split into two bf16 terms, hi = bf16(x) and lo = bf16(x - hi), so |x - hi - lo| <= 2^-16 |x|,
// and the tensor cores accumulate  hi.lo + lo.hi + hi.hi  (three K = 64 products per tile) in fp32.  Error against the
// canonical fp32 score, relative to sum_k |u_k i_k| <= ||u||_2 ||i||_2 (Cauchy-Schwarz):
//   dropped terms (lo.lo and the two residuals)                      <= 3 * 2^-16 * (1 + 2^-7)      = 4.6e-5
//   fp32 accumulation of 12 chained K = 16 MMAs (17 addends each, truncating alignment, 2^-23)  <= 2.5e-5
//   the canonical fp32 chain itself (64 fused multiply-adds, 2^-24)                               <= 0.4e-5
// EV_EPS_REL = 1e-4 covers their sum (7.5e-5) and the rounding of the norms.  eval_rescore_kernel measures the
// largest |approx - exact| / (EV_EPS_REL ||u|| max||i||) it sees into stats[3] (parts per million): tests assert < 1e6.
constexpr float EV_EPS_REL = 1.0e-4f;

enum { EV_SAMPLE = 0, EV_FILTER = 1, EV_FILTER_POOL = 2 };  // EV_FILTER_POOL: the FILTER pass of long lists

struct EvalParams {
    const __nv_bfloat16 *Ap;  // packed test-user rows, [2 terms: hi, lo][n_test_pad / 8][8 chunks][8 rows][8]
    const __nv_bfloat16 *Bp;  // packed item rows,      [2 terms: hi, lo][n_items_pad / 8][...]
    int64_t a_term_stride, b_term_stride;  // bytes between the hi and the lo array
    const int32_t *test_users;
    const int64_t *train_indptr;
    const int32_t *train_indices;
    float *bucket_max;   // SAMPLE out: [n_seg * sub * EV_CSPLIT][n_test_pad][EV_BUCKETS] running maxima of every sample cell
    const float *thr;    // FILTER in:  [n_test_pad] tau - 2 eps (-inf: no bound)
    float2 *cand;        // FILTER out: [sub * EV_CSPLIT][n_test_pad][cap] (approx score, item id bits): one short list per (sub-range, column half, user)
                         // FILTER_POOL out: [n_test_pad][cap], one pool per user
    int32_t *cand_cnt;   // [sub * EV_CSPLIT][n_test_pad]; FILTER_POOL: [n_test_pad] append counters (may run past cap: overflow)
    int32_t *overflow;   // [n_test_pad] flag; [n_test_pad] = count, [n_test_pad + 2 ...] = list of flagged rows
                         // ([n_test_pad + 1] = count, [2 n_test_pad + 2 ...] = rows with more than 256 candidates: eval_rescore_kernel)
    int32_t n_test, n_items, n_tiles;
    // Work decomposition.  The item tiles are cut into n_seg segments (SAMPLE: every segment scores its first seg_tiles tiles;
    // FILTER: one segment = the whole catalogue) of `sub` sub-ranges of sub_tiles tiles; a CELL is (sub-range, 256-user block).
    // The grid is persistent (one CTA per SM); CTA c takes cells c, c + gridDim.x, ...; cells are numbered user-block-minor so
    // that the CTAs running at the same time read the same item tiles (L2 hits, whatever the catalogue size).
    int32_t n_mblk, n_seg, seg_pitch, seg_tiles, sub, sub_tiles;
    int32_t cap;
};

struct EvalCell {
    int m_blk, seg, tile0, n_my;
};
__device__ __forceinline__ EvalCell ev_cell(const EvalParams &P, int w) {
    EvalCell c;
    const int rng = w / P.n_mblk;
    c.m_blk = w - rng * P.n_mblk;
    c.seg = rng / P.sub;
    const int j = rng - c.seg * P.sub;
    c.tile0 = c.seg * P.seg_pitch + j * P.sub_tiles;
    int n = min(P.sub_tiles, P.seg_tiles - j * P.sub_tiles);
    n = min(n, P.n_tiles - c.tile0);
    c.n_my = max(n, 0);
    return c;
}

// ------------------------------------------------------------------------------------------ PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(bar), "r"(bytes)
                 : "memory");
}
// Bounded wait: a protocol bug traps (the launch fails) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done = 0;
    for (uint32_t spins = 0; !done; ++spins) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
        if (!done && spins > (1u << 26)) __trap();
    }
}
__device__ __forceinline__ void bulk_copy_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc], bf16 inputs, fp32 accumulate
__device__ __forceinline__ void tc_mma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tc_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tc_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, no swizzle: 8-row x 16-byte core matrices; LBO = distance between the two core matrices an
// MMA reads along K (128 B), SBO = distance between 8-row groups (1024 B); descriptor version 1 (sm_100).
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(128u >> 4) << 16) | ((uint64_t)(1024u >> 4) << 32) |
           ((uint64_t)1 << 46);
}
// c = f32 (1 << 4), a = b = bf16 (1 << 7, 1 << 10), both K-major, N = 128 (>> 3 at bit 17), M = 128 (>> 4 at bit 24)
constexpr uint32_t EV_IDESC = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(EV_BN >> 3) << 17) | ((128u >> 4) << 24);

// ------------------------------------------------------------------------------------------ 1. pack
// One thread = one (row, 8-element chunk): fp32 -> bf16, written as one 16-byte store into the core-matrix
// layout.  The 8 threads of a row reduce the squared norm; users store 2 * eps, items a global max norm.
__global__ void __launch_bounds__(256) eval_pack_kernel(const float *__restrict__ tab, const int32_t *__restrict__ gather,
                                                        int64_t n_rows, int64_t n_rows_pad, int64_t n_tab_rows,
                                                        __nv_bfloat16 *__restrict__ out, float *__restrict__ row_norm,
                                                        unsigned int *__restrict__ max_norm_bits) {
    const int64_t t = (int64_t)blockIdx.x * 256 + threadIdx.x;
    const int64_t row = t >> 3;
    const int chunk = (int)(t & 7);
    if (row >= n_rows_pad) return;
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
    bool live = row < n_rows;
    if (live) {
        int64_t src = gather ? (int64_t)gather[row] : row;
        if (src < 0 || src >= n_tab_rows) live = false;
        else {
            const float4 *p = reinterpret_cast<const float4 *>(tab + src * EV_D + chunk * 8);
            a = __ldg(p);
            b = __ldg(p + 1);
        }
    }
    const float x[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    __nv_bfloat16 hi[8], lo[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        hi[j] = __float2bfloat16_rn(x[j]);
        lo[j] = __float2bfloat16_rn(x[j] - __bfloat162float(hi[j]));
    }
    const int64_t off = (row >> 3) * 512 + chunk * 64 + (row & 7) * 8;  // in bf16 elements
    *reinterpret_cast<uint4 *>(out + off) = *reinterpret_cast<const uint4 *>(hi);
    *reinterpret_cast<uint4 *>(out + n_rows_pad * EV_D + off) = *reinterpret_cast<const uint4 *>(lo);
    float ss = (a.x * a.x + a.y * a.y) + (a.z * a.z + a.w * a.w) + (b.x * b.x + b.y * b.y) + (b.z * b.z + b.w * b.w);
    ss += __shfl_xor_sync(0xffffffffu, ss, 1);
    ss += __shfl_xor_sync(0xffffffffu, ss, 2);
    ss += __shfl_xor_sync(0xffffffffu, ss, 4);
    if (chunk == 0) {
        const float nrm = sqrtf(ss) * 1.0001f;
        if (row_norm) row_norm[row] = live ? nrm : 0.f;
        if (max_norm_bits && live) atomicMax(max_norm_bits, __float_as_uint(nrm));  // nrm >= 0: bit order = value order
    }
}

// slack[row] = 2 * eps = 2 * EV_EPS_REL * ||u|| * max ||i||
__global__ void eval_slack_kernel(float *__restrict__ slack, int64_t n, const unsigned int *__restrict__ max_norm_bits) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r < n) slack[r] = 2.0f * EV_EPS_REL * slack[r] * __uint_as_float(*max_norm_bits) + 1e-30f;
}

// ------------------------------------------------------------------------------------------ 2. scores
struct EvalSmem {
    // offsets into dynamic shared memory (base aligned to 1024)
    static constexpr int A = 0;                      // [hi 32 KB | lo 32 KB]
    static constexpr int B = A + 2 * EV_A_BYTES;     // per stage [hi 16 KB | lo 16 KB]
    static constexpr int END = B + EV_STAGES * 2 * EV_B_BYTES;
};

// Bit j = column col0 + j is one of the user's training items (or, in the last tile, a padding column).  nt0 / nt1 are the next
// two training items of the row (software-pipelined: the load of nt1 is in flight while nt0 is used).
__device__ __forceinline__ unsigned ev_train_mask(int col0, int n_items, int &nt0, int &nt1, int64_t &tp, int64_t tend,
                                                  const int32_t *__restrict__ train_indices) {
    unsigned mb = 0;
    if (nt0 < col0 + 32) {
        do {
            if (nt0 >= col0) mb |= 1u << (nt0 - col0);  // items below col0 lie in columns another warp examines
            nt0 = nt1;
            ++tp;
            nt1 = tp + 1 < tend ? __ldg(train_indices + tp + 1) : INT_MAX;
        } while (nt0 < col0 + 32);
    }
    if (col0 + 32 > n_items) mb |= (col0 >= n_items) ? 0xffffffffu : (0xffffffffu << (n_items - col0));
    return mb;
}

// SAMPLE: the masked columns become NaN (NaN never compares >= a threshold and fmaxf ignores it) before the running maxima.
__device__ __forceinline__ void ev_poison(uint32_t (&v)[32], unsigned mb) {
    if (mb) {
#pragma unroll
        for (int j = 0; j < 32; ++j)
            if (mb & (1u << j)) v[j] = 0x7fc00000u;
    }
}

// Append the columns of one 4-column group that meet the user's threshold to THIS THREAD's candidate list: every
// (sub-range of the catalogue, column half, user row) owns a short list of `cap` slots, so the hot path needs no atomics and
// no hand-over -- plain stores at a private counter.  (Tried and dropped in round 2: one list per user with slots handed out by
// global atomicAdd, directly or through a per-warp shared-memory ring drained one tile later: the scoring pass is bound by
// the instructions its 16 epilogue warps issue, 7 300 -> 11 200 warp instructions per tile, 2.2 -> 2.8 ms at the Amazon-Book
// shape.)  Branch-free: the four slots are computed up front and the stores are predicated.
// `masked`: bit q = column col + q is a training item / padding column and is never appended (the FILTER pass does not turn them
// into NaN first: that 32-way select ran whenever ANY lane of the warp had a training item in the chunk, half of all chunks at
// the Amazon-Book shape; here the mask costs four bit tests on the rare path).
__device__ __noinline__ int ev_append4(float x0, float x1, float x2, float x3, float thr, int col, int cnt, int cap,
                                       float2 *__restrict__ crow, unsigned masked) {
    const bool h0 = x0 >= thr && !(masked & 1u), h1 = x1 >= thr && !(masked & 2u), h2 = x2 >= thr && !(masked & 4u),
               h3 = x3 >= thr && !(masked & 8u);
    const int c0 = cnt, c1 = c0 + (h0 ? 1 : 0), c2 = c1 + (h1 ? 1 : 0), c3 = c2 + (h2 ? 1 : 0);
    if (h0 && c0 < cap) crow[c0] = make_float2(x0, __int_as_float(col));
    if (h1 && c1 < cap) crow[c1] = make_float2(x1, __int_as_float(col + 1));
    if (h2 && c2 < cap) crow[c2] = make_float2(x2, __int_as_float(col + 2));
    if (h3 && c3 < cap) crow[c3] = make_float2(x3, __int_as_float(col + 3));
    return c3 + (h3 ? 1 : 0);
}

template <int MODE>
__global__ void __launch_bounds__(EV_THREADS, 1) eval_scores_kernel(const EvalParams P) {
    extern __shared__ uint8_t ev_smem_raw[];
    const uint32_t raw = smem_u32(ev_smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;  // 1024-byte aligned view of dynamic shared memory
    __shared__ __align__(8) uint64_t bars[2 * EV_STAGES + 2 + 8];
    __shared__ uint32_t tmem_base_slot;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_cells = P.n_mblk * P.n_seg * P.sub;

    const uint32_t bar_full = smem_u32(&bars[0]);               // [EV_STAGES] item tile landed
    const uint32_t bar_empty = smem_u32(&bars[EV_STAGES]);      // [EV_STAGES] item tile consumed by the MMAs
    const uint32_t bar_a_full = smem_u32(&bars[2 * EV_STAGES]);       // user block of the current cell landed
    const uint32_t bar_a_empty = smem_u32(&bars[2 * EV_STAGES + 1]);  // every MMA of the current cell has read it
    // accumulator hand-over per (stage, 128-row half): the epilogue warps of a half start as soon as ITS 12 MMAs are done and
    // the MMAs of a half restart as soon as ITS 8 warps have drained it (per-tile barriers: 3 450 clocks per tile, these: see profiles/eval_r2.md)
    const uint32_t bar_tfull = smem_u32(&bars[2 * EV_STAGES + 2]);   // [2 stages][2 halves] accumulators ready
    const uint32_t bar_tempty = smem_u32(&bars[2 * EV_STAGES + 6]);  // [2 stages][2 halves] accumulators drained by the epilogue

    if (threadIdx.x == 0) {
        for (int s = 0; s < EV_STAGES; ++s) {
            mbar_init(bar_full + 8 * s, 1);
            mbar_init(bar_empty + 8 * s, 1);
        }
        mbar_init(bar_a_full, 1);
        mbar_init(bar_a_empty, 1);
        for (int s = 0; s < 4; ++s) {
            mbar_init(bar_tfull + 8 * s, 1);
            mbar_init(bar_tempty + 8 * s, EV_EPI_WARPS / 2);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {  // TMEM allocation is a warp-wide operation; the same warp frees it
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_slot)),
                     "r"((uint32_t)EV_TMEM_COLS)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_slot;

    // Every role walks the same cell list (ev_cell is a pure function of the cell number); `git` counts the item tiles this
    // CTA has been through, so the shared-memory ring and the two accumulator stages keep their phases across cells; `wi`
    // counts its non-empty cells (phases of the user-block barriers).
    if (warp == 0) {
        // ===== producer: two 32 KB bulk copies per cell for the user block (hi, lo), two 16 KB bulk copies per item tile =====
        if (lane == 0) {
            uint32_t git = 0, wi = 0;
            const uint8_t *b_src = reinterpret_cast<const uint8_t *>(P.Bp);
            for (int w = blockIdx.x; w < n_cells; w += gridDim.x) {
                const EvalCell c = ev_cell(P, w);
                if (c.n_my == 0) continue;
                const uint8_t *a_src = reinterpret_cast<const uint8_t *>(P.Ap) + (int64_t)c.m_blk * EV_A_BYTES;
                mbar_wait(bar_a_empty, (wi & 1) ^ 1);  // the previous cell's MMAs are done with the user block
                mbar_arrive_expect_tx(bar_a_full, 2 * EV_A_BYTES);
                bulk_copy_g2s(base + EvalSmem::A, a_src, EV_A_BYTES, bar_a_full);
                bulk_copy_g2s(base + EvalSmem::A + EV_A_BYTES, a_src + P.a_term_stride, EV_A_BYTES, bar_a_full);
                ++wi;
                for (int it = 0; it < c.n_my; ++it, ++git) {
                    const int s = git % EV_STAGES;
                    const uint32_t ph = (git / EV_STAGES) & 1;
                    mbar_wait(bar_empty + 8 * s, ph ^ 1);
                    mbar_arrive_expect_tx(bar_full + 8 * s, 2 * EV_B_BYTES);
                    const uint32_t dst = base + EvalSmem::B + s * 2 * EV_B_BYTES;
                    const uint8_t *src = b_src + (int64_t)(c.tile0 + it) * EV_B_BYTES;
                    bulk_copy_g2s(dst, src, EV_B_BYTES, bar_full + 8 * s);
                    bulk_copy_g2s(dst + EV_B_BYTES, src + P.b_term_stride, EV_B_BYTES, bar_full + 8 * s);
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: one thread =====
        if (lane == 0) {
            uint32_t git = 0, wi = 0;
            for (int w = blockIdx.x; w < n_cells; w += gridDim.x) {
                const EvalCell c = ev_cell(P, w);
                if (c.n_my == 0) continue;
                mbar_wait(bar_a_full, wi & 1);
                ++wi;
                for (int it = 0; it < c.n_my; ++it, ++git) {
                    const int s = git % EV_STAGES;
                    const uint32_t ph = (git / EV_STAGES) & 1;
                    const int as = git & 1;
                    const uint32_t aph = (git >> 1) & 1;
                    mbar_wait(bar_full + 8 * s, ph);          // item tile landed
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        mbar_wait(bar_tempty + 8 * (as * 2 + h), aph ^ 1);  // the epilogue drained this half of the accumulator stage
                        tc_fence_after();
                        const uint32_t d = tmem_base + (uint32_t)(as * 256 + h * 128);
                        const uint32_t a_hi = base + EvalSmem::A + h * (EV_A_BYTES / 2), a_lo = a_hi + EV_A_BYTES;
                        const uint32_t b_hi = base + EvalSmem::B + s * 2 * EV_B_BYTES, b_lo = b_hi + EV_B_BYTES;
                        // small terms first: hi.lo, lo.hi, then hi.hi
#pragma unroll
                        for (int t = 0; t < 3; ++t) {
                            const uint32_t a_t = t == 1 ? a_lo : a_hi;
                            const uint32_t b_t = t == 0 ? b_lo : b_hi;
#pragma unroll
                            for (int k = 0; k < EV_D / 16; ++k)
                                tc_mma_bf16(d, umma_desc(a_t + k * 256), umma_desc(b_t + k * 256), EV_IDESC, (t | k) ? 1u : 0u);
                        }
                        tc_commit(bar_tfull + 8 * (as * 2 + h));  // this half's accumulators are ready for its 8 epilogue warps
                    }
                    tc_commit(bar_empty + 8 * s);    // smem slot reusable once these MMAs have read it
                }
                tc_commit(bar_a_empty);  // the user block may be overwritten once every MMA of this cell has completed
            }
        }
    } else {
        // ===== epilogue: 16 warps; thread = one user row of one 128-row half x one 64-column half of every tile =====
        const int ew = warp - 2;
        const int quad = warp & 3;  // TMEM lane quadrant this warp may read
        const int half = (ew >> 2) & 1;
        const int chalf = ew >> 3;
        const int64_t n_pad = (int64_t)P.n_mblk * EV_BM;
        uint32_t git = 0;
        float bm[EV_BUCKETS];  // SAMPLE: running maxima of the cell, bucket = column mod 32
        for (int w = blockIdx.x; w < n_cells; w += gridDim.x) {
            const EvalCell c = ev_cell(P, w);
            if (c.n_my == 0) continue;
            const int64_t row = (int64_t)c.m_blk * EV_BM + half * 128 + quad * 32 + lane;
            const bool live = row < P.n_test;
            // training items of this user at or after the cell's first column, walked in step with the columns
            int64_t tp = 0, tend = 0;
            if (live) {
                const int32_t u = P.test_users[row];
                tp = P.train_indptr[u];
                tend = P.train_indptr[u + 1];
                const int first_col = c.tile0 * EV_BN;
                int64_t lo = tp, hi = tend;
                while (lo < hi) {
                    const int64_t mid = (lo + hi) >> 1;
                    if (P.train_indices[mid] < first_col) lo = mid + 1;
                    else hi = mid;
                }
                tp = lo;
            }
            int nt0 = tp < tend ? __ldg(P.train_indices + tp) : INT_MAX;
            int nt1 = tp + 1 < tend ? __ldg(P.train_indices + tp + 1) : INT_MAX;
#pragma unroll
            for (int j = 0; j < EV_BUCKETS; ++j) bm[j] = -CUDART_INF_F;
            float thr = CUDART_INF_F;  // FILTER: fixed threshold of this user (a dead row never appends)
            int cnt = 0;
            float2 *crow = nullptr;
            const int rng = w / P.n_mblk;                  // sub-range of the catalogue this cell scores
            const int part = rng * EV_CSPLIT + chalf;      // slice of the candidate / bucket arrays this thread fills
            if (MODE == EV_FILTER) {
                if (live) thr = P.thr[row];
                crow = P.cand + ((int64_t)part * n_pad + row) * P.cap;
            }
            if (MODE == EV_FILTER_POOL) {
                if (live) thr = P.thr[row];
                crow = P.cand + row * P.cap;
            }

            for (int it = 0; it < c.n_my; ++it, ++git) {
                const int as = git & 1;
                const uint32_t aph = (git >> 1) & 1;
                mbar_wait(bar_tfull + 8 * (as * 2 + half), aph);
                tc_fence_after();
                const uint32_t tcol = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(as * 256 + half * 128);
                const int col_tile = (c.tile0 + it) * EV_BN;
                // this warp's 64 columns of the tile as two 32-column TMEM loads; four epilogue warps per scheduler hide
                // the load latency, so there is a single register buffer (the kernel must stay under 112 registers)
#pragma unroll 1
                for (int cc = 0; cc < 2; ++cc) {
                    const int cq = chalf * 2 + cc;
                    uint32_t v[32];
                    tc_ld32(tcol + cq * 32, v);
                    tc_ld_wait();
                    const int col0 = col_tile + cq * 32;
                    unsigned mb = 0;
                    if (nt0 < col0 + 32 || col0 + 32 > P.n_items) mb = ev_train_mask(col0, P.n_items, nt0, nt1, tp, tend, P.train_indices);
                    if (MODE == EV_SAMPLE) {
                        ev_poison(v, mb);
#pragma unroll
                        for (int j = 0; j < 32; ++j) bm[j] = fmaxf(bm[j], __uint_as_float(v[j]));
                    } else {
                        // group maxima first (over the RAW scores: a masked column that meets the threshold only costs a visit
                        // of the rare path, where its mask bit keeps it out): a user row meets its threshold in ~1 of 30 chunks,
                        // and then usually in a single group of 4 columns
                        float m4[8];
#pragma unroll
                        for (int g = 0; g < 8; ++g)
                            m4[g] = fmaxf(fmaxf(__uint_as_float(v[4 * g]), __uint_as_float(v[4 * g + 1])),
                                          fmaxf(__uint_as_float(v[4 * g + 2]), __uint_as_float(v[4 * g + 3])));
                        const float m = fmaxf(fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3])),
                                              fmaxf(fmaxf(m4[4], m4[5]), fmaxf(m4[6], m4[7])));
                        if (MODE == EV_FILTER && m >= thr) {
#pragma unroll
                            for (int g = 0; g < 8; ++g)
                                if (m4[g] >= thr)
                                    cnt = ev_append4(__uint_as_float(v[4 * g]), __uint_as_float(v[4 * g + 1]), __uint_as_float(v[4 * g + 2]),
                                                     __uint_as_float(v[4 * g + 3]), thr, col0 + 4 * g, cnt, P.cap, crow, (mb >> (4 * g)) & 15u);
                        }
                        if (MODE == EV_FILTER_POOL && m >= thr) {
                            // long lists: the chunk's hits take their slots of the user's pool with ONE atomicAdd (the lanes of a
                            // warp issue theirs together), so a warp waits for at most one round trip per 32 columns
                            unsigned hm = 0;
#pragma unroll
                            for (int j = 0; j < 32; ++j) hm |= (__uint_as_float(v[j]) >= thr ? 1u : 0u) << j;
                            hm &= ~mb;
                            if (hm) {
                                const int n = __popc(hm);
                                int slot = atomicAdd(P.cand_cnt + row, n);
                                if (slot + n > P.cap && slot <= P.cap && atomicExch(P.overflow + row, 1) == 0)  // this append crosses the end
                                    P.overflow[n_pad + 2 + atomicAdd(P.overflow + n_pad, 1)] = (int32_t)row;
                                if (slot < P.cap) {
#pragma unroll
                                    for (int g = 0; g < 8; ++g)
                                        if ((hm >> (4 * g)) & 15u)
                                            slot = ev_append4(__uint_as_float(v[4 * g]), __uint_as_float(v[4 * g + 1]), __uint_as_float(v[4 * g + 2]),
                                                              __uint_as_float(v[4 * g + 3]), thr, col0 + 4 * g, slot, P.cap, crow, (mb >> (4 * g)) & 15u);
                                }
                            }
                        }
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_tempty + 8 * (as * 2 + half));
            }
            if (MODE == EV_SAMPLE && live) {
                // every cell (segment, sub-range, column half) owns its 32 buckets: plain stores (the first version merged the
                // sub-ranges of a segment with atomicMax: 40 M reductions, +150 us at the Amazon-Book shape)
                float4 *o = reinterpret_cast<float4 *>(P.bucket_max + ((int64_t)part * n_pad + row) * EV_BUCKETS);
#pragma unroll
                for (int j = 0; j < EV_BUCKETS / 4; ++j) o[j] = make_float4(bm[4 * j], bm[4 * j + 1], bm[4 * j + 2], bm[4 * j + 3]);
            }
            if (MODE == EV_FILTER && live) {
                P.cand_cnt[(int64_t)part * n_pad + row] = min(cnt, P.cap);
                if (cnt > P.cap && atomicExch(P.overflow + row, 1) == 0) P.overflow[n_pad + 2 + atomicAdd(P.overflow + n_pad, 1)] = (int32_t)row;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)EV_TMEM_COLS)
                     : "memory");
    }
}

// ------------------------------------------------------------------------------------------ exact helpers
__device__ __forceinline__ uint32_t orderable(float s) {
    if (s == 0.f) s = 0.f;  // -0 and +0 tie
    const uint32_t b = __float_as_uint(s);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
// larger key = better: score descending, then item id ascending
__device__ __forceinline__ unsigned long long rank_key(float s, int id) {
    return ((unsigned long long)orderable(s) << 32) | (unsigned long long)(0xffffffffu - (uint32_t)id);
}
__device__ __forceinline__ unsigned long long warp_max_u64(unsigned long long k) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, k, o);
        k = other > k ? other : k;
    }
    return k;
}
// canonical score: ascending-k fused multiply-add chain (oracle/hgr_oracle.c hgr_oracle_scores_f32)
__device__ __forceinline__ float exact_score(const float *__restrict__ u_sm, const float *__restrict__ item_row, int D) {
    float acc = 0.f;
    const float4 *p = reinterpret_cast<const float4 *>(item_row);
    for (int k = 0; k < D / 4; ++k) {
        const float4 q = __ldg(p + k);
        acc = fmaf(u_sm[4 * k], q.x, acc);
        acc = fmaf(u_sm[4 * k + 1], q.y, acc);
        acc = fmaf(u_sm[4 * k + 2], q.z, acc);
        acc = fmaf(u_sm[4 * k + 3], q.w, acc);
    }
    return acc;
}
__device__ __forceinline__ bool is_train_item(const int32_t *__restrict__ a, int64_t lo, int64_t hi, int v) {
    const int64_t end = hi;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (__ldg(a + mid) < v) lo = mid + 1;
        else hi = mid;
    }
    return lo < end && __ldg(a + lo) == v;
}
// Block-wide bitonic sort of n (a power of two) keys in shared memory, largest first.  The whole block calls it after a
// __syncthreads() that publishes the keys; it returns after one that publishes the result.
__device__ __forceinline__ void block_sort_desc(unsigned long long *a, int n) {
    for (int k = 2; k <= n; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int p = threadIdx.x; p < n / 2; p += blockDim.x) {
                const int i = ((p & ~(j - 1)) << 1) | (p & (j - 1));  // the lower element of the p-th pair, partner i + j
                const unsigned long long x = a[i], y = a[i + j];
                if ((i & k) == 0 ? x < y : x > y) {  // descending runs where bit k of i is clear
                    a[i] = y;
                    a[i + j] = x;
                }
            }
            __syncthreads();
        }
    }
}

// ------------------------------------------------------------------------------------------ tau
// One warp per test user: tau = K-th largest of the n_seg * 32 bucket maxima of the sample pass.  Every bucket
// maximum is the score of a distinct unmasked item, so at least K items score >= tau: tau is a lower bound of
// the user's K-th best approximate score.  Fewer than K non-empty buckets: no bound (-inf).
// thr = tau - 2 eps with eps = EV_EPS_REL * ||u|| * max ||i|| (see EV_EPS_REL).
// LONG (64 < K <= 256): no merging -- up to 16 keys per lane, 512 bucket maxima >= 2 K -- and the K-th largest key is built
// bit by bit (the largest t that at least K keys reach; keys are unique, so t is one of them): 64 warp-wide counts, not K rounds.
template <bool LONG>
__global__ void __launch_bounds__(128) eval_tau_kernel(const float *__restrict__ bucket_max, int n_seg, int64_t n_pad, int n_test,
                                                       int K, const float *__restrict__ slack, float *__restrict__ thr) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * 4 + warp;
    if (row >= n_test) return;
    if constexpr (LONG) {
        unsigned long long keys[16];
#pragma unroll
        for (int s = 0; s < 16; ++s) {
            const float v = s < n_seg ? bucket_max[((int64_t)s * n_pad + row) * EV_BUCKETS + lane] : -CUDART_INF_F;
            keys[s] = v > -CUDART_INF_F ? rank_key(v, s * EV_BUCKETS + lane) : 0ull;  // 0: empty bucket (or NaN), never counted
        }
        unsigned long long t = 0ull;
        for (int b = 63; b >= 0; --b) {
            const unsigned long long c = t | (1ull << b);
            unsigned n = 0;
#pragma unroll
            for (int s = 0; s < 16; ++s) n += keys[s] >= c;
            if (__reduce_add_sync(0xffffffffu, n) >= (unsigned)K) t = c;
        }
        if (lane == 0) {
            float tau = -CUDART_INF_F;  // t == 0: fewer than K non-empty buckets
            if (t != 0ull) {
                const uint32_t ob = (uint32_t)(t >> 32);
                tau = __uint_as_float((ob & 0x80000000u) ? (ob & 0x7fffffffu) : ~ob);
            }
            thr[row] = tau - slack[row];
        }
        return;
    }
    // Up to 16 bucket maxima per lane are merged down to 4 (the maximum of a group of buckets is the score of one
    // item of the union bucket): 128 disjoint buckets over the whole sample, a K-th largest within 1-2 ranks of the one
    // over 512 buckets at a quarter of the selection work.
    const int per = (n_seg + 3) / 4;
    unsigned long long keys[4] = {0ull, 0ull, 0ull, 0ull};
#pragma unroll
    for (int s = 0; s < 16; ++s) {
        if (s < n_seg) {
            const float v = bucket_max[((int64_t)s * n_pad + row) * EV_BUCKETS + lane];
            if (v > -CUDART_INF_F) {  // false for NaN and for empty buckets
                const unsigned long long k = rank_key(v, s * EV_BUCKETS + lane);
                const int q = s / per;
#pragma unroll
                for (int m = 0; m < 4; ++m)
                    if (m == q && k > keys[m]) keys[m] = k;
            }
        }
    }
    unsigned long long prev = ~0ull, best = 0ull;
    for (int r = 0; r < K; ++r) {
        best = 0ull;
#pragma unroll
        for (int m = 0; m < 4; ++m)
            if (keys[m] < prev && keys[m] > best) best = keys[m];
        best = warp_max_u64(best);
        if (best == 0ull) break;
        prev = best;
    }
    if (lane == 0) {
        float tau = -CUDART_INF_F;
        if (best != 0ull) {
            const uint32_t ob = (uint32_t)(best >> 32);
            tau = __uint_as_float((ob & 0x80000000u) ? (ob & 0x7fffffffu) : ~ob);
        }
        thr[row] = tau - slack[row];
    }
}

// ------------------------------------------------------------------------------------------ 3. rescore
constexpr int RS_WARPS = 4;
constexpr int RS_CAP = 1024;  // candidates of one user held in shared memory
constexpr int RS_POOL_MAX = 2048;  // long lists: largest pool of one user (EV_POOL_PER_K * EV_MAX_K), sorted by one block
constexpr int RS_POOL_WARPS = 8;

// stats of one user's re-scoring: candidates, survivors, and the observed error in parts per million of the bound
// eps = slack / 2 (must stay below 1e6)
__device__ __forceinline__ void rs_add_stats(unsigned long long *__restrict__ stats, int n_c, int n_keep, float worst, float slack) {
    atomicAdd(stats + 0, (unsigned long long)n_c);
    atomicAdd(stats + 1, (unsigned long long)n_keep);
    atomicMax(stats + 3, (unsigned long long)(worst / (0.5f * slack) * 1.0e6f));
}
// fewer than K unmasked items in the whole catalogue: the reference then returns masked items (-10e8) in ascending id order
// (oracle topk_exact keeps them as candidates).  Positions filled .. K-1 of the row, thread t of `step` takes t, t + step, ...
__device__ __forceinline__ void rs_fill_masked(const int64_t *__restrict__ train_indptr, const int32_t *__restrict__ train_indices,
                                               int32_t u, int64_t row, int K, int filled, int t, int step, int32_t *__restrict__ out_ids,
                                               float *__restrict__ out_scores) {
    const int64_t t0 = train_indptr[u], t1 = train_indptr[u + 1];
    for (int r = filled + t; r < K; r += step) {
        const int64_t q = t0 + (r - filled);
        out_ids[row * K + r] = q < t1 ? train_indices[q] : -1;
        out_scores[row * K + r] = EV_MASK_SCORE;
    }
}

// One warp per test user.  (a) the candidates' approximate scores give the approximate K-th best tau_a;
// (b) candidates below tau_a - 2 eps cannot be in the exact top-K and are dropped; (c) the survivors are
// re-scored exactly; (d) K rounds of warp arg-max on (score desc, id asc) keys.
// Two launches share the users: CAP = 256 (most users: 2 KB of keys per warp, 64 registers, 8 blocks per SM -- the kernel is a chain
// of dependent memory round trips per warp, so resident warps are what it needs) takes the lists of up to 256 candidates and
// lists the rows with more; the CAP = RS_CAP launch (LO >= 0) walks that list.
// UW > 1 (long lists): one block of UW warps per user, whose pool of up to CAP candidates (the plan's cap, rounded up to a power of
// two, of dynamic shared memory) is sorted by (a) approximate and (d) exact key with a block-wide bitonic sort: after the first sort
// the K-th best is keys[K - 1] and the survivors of (b) are a prefix, so no step takes K dependent rounds.
template <int CAP, int LO, int MINB, int UW = 1>
__global__ void __launch_bounds__(UW > 1 ? UW * 32 : RS_WARPS * 32, MINB) eval_rescore_kernel(
    const float *__restrict__ user_emb, const float *__restrict__ item_emb, int D, const int32_t *__restrict__ test_users,
    const int64_t *__restrict__ train_indptr, const int32_t *__restrict__ train_indices, const float2 *__restrict__ cand,
    const int32_t *__restrict__ cand_cnt, const float *__restrict__ slack, int32_t *__restrict__ overflow, int n_parts,
    int64_t n_pad, int cap, int n_test, int K, int32_t *__restrict__ out_ids, float *__restrict__ out_scores,
    unsigned long long *__restrict__ stats) {
    __shared__ float u_sm[RS_WARPS][128];
    __shared__ unsigned long long keys[RS_WARPS][UW > 1 ? 1 : CAP];  // UW > 1: the keys live in dynamic shared memory
    if constexpr (UW > 1) {
        extern __shared__ unsigned long long pool[];
        __shared__ int s_keep;
        __shared__ unsigned s_worst;
        const int64_t row = blockIdx.x;
        if (row >= n_test || overflow[row]) return;  // overflowed pools are handled by eval_brute_kernel
        const int n_c = min(cand_cnt[row], cap);
        const int32_t u = test_users[row];
        for (int k = threadIdx.x; k < D; k += UW * 32) u_sm[0][k] = user_emb[(int64_t)u * D + k];
        int n_pow = 1;
        while (n_pow < n_c) n_pow <<= 1;
        // (a) approximate keys, padded with 0 (below every key) to a power of two, sorted best first
        const float2 *lst = cand + row * cap;
        for (int j = threadIdx.x; j < n_pow; j += UW * 32) {
            unsigned long long k = 0ull;
            if (j < n_c) {
                const float2 c = lst[j];
                k = rank_key(c.x, __float_as_int(c.y));
            }
            pool[j] = k;
        }
        if (threadIdx.x == 0) {
            s_keep = 0;
            s_worst = 0u;
        }
        __syncthreads();
        block_sort_desc(pool, n_pow);
        // (b) keep keys >= (tau_a - 2 eps), tau_a = the K-th best approximate score: a prefix of the sorted pool
        unsigned long long keep_key = 0ull;
        if (n_c >= K) {
            const uint32_t ob = (uint32_t)(pool[K - 1] >> 32);
            const float tau_a = __uint_as_float((ob & 0x80000000u) ? (ob & 0x7fffffffu) : ~ob);
            keep_key = (unsigned long long)orderable(tau_a - slack[row]) << 32;
        }
        for (int j = threadIdx.x; j < n_c; j += UW * 32)
            if (pool[j] >= keep_key && (j + 1 == n_c || pool[j + 1] < keep_key)) s_keep = j + 1;
        __syncthreads();
        const int n_keep = s_keep;
        // (c) exact re-scoring in place; the slots up to the next power of two are cleared for the second sort
        int n_pow2 = 1;
        while (n_pow2 < n_keep) n_pow2 <<= 1;
        float worst = 0.f;
        for (int j = threadIdx.x; j < n_pow2; j += UW * 32) {
            unsigned long long nk = 0ull;
            if (j < n_keep) {
                const unsigned long long k = pool[j];
                const int id = (int32_t)(0xffffffffu - (uint32_t)(k & 0xffffffffu));
                const float ex = exact_score(u_sm[0], item_emb + (int64_t)id * D, D);
                const uint32_t ob = (uint32_t)(k >> 32);
                worst = fmaxf(worst, fabsf(__uint_as_float((ob & 0x80000000u) ? (ob & 0x7fffffffu) : ~ob) - ex));
                nk = rank_key(ex, id);
            }
            pool[j] = nk;
        }
        if (worst > 0.f) atomicMax(&s_worst, __float_as_uint(worst));  // worst >= 0: bit order = value order
        __syncthreads();
        // (d) exact top-K
        block_sort_desc(pool, n_pow2);
        const int filled = n_keep < K ? n_keep : K;
        for (int r = threadIdx.x; r < filled; r += UW * 32) {
            const unsigned long long k = pool[r];
            const uint32_t ob = (uint32_t)(k >> 32);
            out_ids[row * K + r] = (int32_t)(0xffffffffu - (uint32_t)(k & 0xffffffffu));
            out_scores[row * K + r] = __uint_as_float((ob & 0x80000000u) ? (ob & 0x7fffffffu) : ~ob);
        }
        if (threadIdx.x == 0 && stats) rs_add_stats(stats, n_c, n_keep, __uint_as_float(s_worst), slack[row]);
        rs_fill_masked(train_indptr, train_indices, u, row, K, filled, threadIdx.x, UW * 32, out_ids, out_scores);
        return;
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int64_t row = (int64_t)blockIdx.x * RS_WARPS + warp;
    if (LO >= 0) {  // second launch: the rows the first one listed (one block per RS_WARPS of them; the rest of the grid leaves)
        if (row >= overflow[n_pad + 1]) return;
        row = overflow[2 * n_pad + 2 + row];
    }
    if (row >= n_test) return;
    if (overflow[row]) return;  // handled by eval_brute_kernel
    // list lengths of up to 64 parts, one or two per lane (read once; the copy loop below gets them by shuffle)
    const int cnt_a = lane < n_parts ? cand_cnt[(int64_t)lane * n_pad + row] : 0;
    const int cnt_b = lane + 32 < n_parts ? cand_cnt[(int64_t)(lane + 32) * n_pad + row] : 0;
    int n_c = cnt_a + cnt_b;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) n_c += __shfl_xor_sync(0xffffffffu, n_c, o);
    if (n_c > CAP) {
        if (lane == 0) {
            if (CAP < RS_CAP && n_c <= RS_CAP) overflow[2 * n_pad + 2 + atomicAdd(overflow + n_pad + 1, 1)] = (int32_t)row;  // second launch
            else if (atomicExch(overflow + row, 1) == 0) overflow[n_pad + 2 + atomicAdd(overflow + n_pad, 1)] = (int32_t)row;
        }
        return;
    }
    const int32_t u = test_users[row];
    for (int k = lane; k < D; k += 32) u_sm[warp][k] = user_emb[(int64_t)u * D + k];
    // (a) approximate keys into shared memory
    // lane l copies list l (and list l + 32): every lane walks its own short list, so all lists are read concurrently -- two
    // memory round trips for the whole row (one list after the other, 24 lists: 0.2 ms more at the Amazon-Book shape)
    {
        int inc = cnt_a;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += v;
        }
        const int total_a = __shfl_sync(0xffffffffu, inc, 31);
        int off_a = inc - cnt_a;
        int incb = cnt_b;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incb, o);
            if (lane >= o) incb += v;
        }
        int off_b = total_a + incb - cnt_b;
        const float2 *la = cand + ((int64_t)lane * n_pad + row) * cap;
        for (int j = 0; j < cnt_a; j += 4) {
            float2 c[4];
#pragma unroll
            for (int q = 0; q < 4; ++q)
                if (j + q < cnt_a) c[q] = la[j + q];
#pragma unroll
            for (int q = 0; q < 4; ++q)
                if (j + q < cnt_a) keys[warp][off_a + j + q] = rank_key(c[q].x, __float_as_int(c[q].y));
        }
        if (cnt_b > 0) {
            const float2 *lb = cand + ((int64_t)(lane + 32) * n_pad + row) * cap;
            for (int j = 0; j < cnt_b; ++j) {
                const float2 c = lb[j];
                keys[warp][off_b + j] = rank_key(c.x, __float_as_int(c.y));
            }
        }
    }
    __syncwarp();
    // K-th best approximate key.  Small lists (the usual case): every lane counts how many keys beat each of its own
    // (keys are unique: the id is part of the key), the key beaten by exactly K - 1 others is the answer.
    unsigned long long prev = ~0ull, best = 0ull;
    if (CAP <= 256 || n_c <= 256) {
        unsigned long long mine[8];
        int beat[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            mine[q] = lane + 32 * q < n_c ? keys[warp][lane + 32 * q] : 0ull;
            beat[q] = 0;
        }
        for (int j = 0; j < n_c; ++j) {
            const unsigned long long k = keys[warp][j];  // broadcast read
#pragma unroll
            for (int q = 0; q < 8; ++q) beat[q] += k > mine[q];
        }
        unsigned long long kth = 0ull;
#pragma unroll
        for (int q = 0; q < 8; ++q)
            if (lane + 32 * q < n_c && beat[q] == K - 1) kth = mine[q];
        best = warp_max_u64(kth);  // 0 when the list holds fewer than K keys
    } else {
        for (int r = 0; r < K; ++r) {
            best = 0ull;
            for (int j = lane; j < n_c; j += 32) {
                const unsigned long long k = keys[warp][j];
                if (k < prev && k > best) best = k;
            }
            best = warp_max_u64(best);
            if (best == 0ull) break;
            prev = best;
        }
    }
    // (b) + (c): keep keys >= (tau_a - 2 eps), re-score them, compact in place (slot <= source index)
    unsigned long long keep_key = 0ull;
    if (best != 0ull) {
        const uint32_t ob = (uint32_t)(best >> 32);
        const float tau_a = __uint_as_float((ob & 0x80000000u) ? (ob & 0x7fffffffu) : ~ob);
        keep_key = (unsigned long long)orderable(tau_a - slack[row]) << 32;
    }
    int n_keep = 0;
    float worst = 0.f;  // largest |approximate - exact| among the re-scored candidates
    for (int j0 = 0; j0 < n_c; j0 += 32) {
        const int j = j0 + lane;
        bool ok = false;
        unsigned long long nk = 0ull;
        if (j < n_c) {
            const unsigned long long k = keys[warp][j];
            ok = k >= keep_key;
            if (ok) {
                const int id = (int32_t)(0xffffffffu - (uint32_t)(k & 0xffffffffu));
                const float ex = exact_score(u_sm[warp], item_emb + (int64_t)id * D, D);
                const uint32_t ob = (uint32_t)(k >> 32);
                worst = fmaxf(worst, fabsf(__uint_as_float((ob & 0x80000000u) ? (ob & 0x7fffffffu) : ~ob) - ex));
                nk = rank_key(ex, id);
            }
        }
        const unsigned m = __ballot_sync(0xffffffffu, ok);
        __syncwarp();
        if (ok) keys[warp][n_keep + __popc(m & ((1u << lane) - 1u))] = nk;
        n_keep += __popc(m);
        __syncwarp();
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) worst = fmaxf(worst, __shfl_xor_sync(0xffffffffu, worst, o));
    if (lane == 0 && stats) rs_add_stats(stats, n_c, n_keep, worst, slack[row]);
    // (d) exact top-K.  Few survivors (the usual case): the rank of a key = the number of keys that beat it = its
    // position in the list; otherwise K rounds of "best key strictly below the previous winner".
    int filled = 0;
    if (n_keep <= 64) {
        __syncwarp();
        const unsigned long long m0 = lane < n_keep ? keys[warp][lane] : 0ull;
        const unsigned long long m1 = lane + 32 < n_keep ? keys[warp][lane + 32] : 0ull;
        int b0 = 0, b1 = 0;
        for (int j = 0; j < n_keep; ++j) {
            const unsigned long long k = keys[warp][j];
            b0 += k > m0;
            b1 += k > m1;
        }
        if (lane < n_keep && b0 < K) {
            const uint32_t ob = (uint32_t)(m0 >> 32);
            out_ids[row * K + b0] = (int32_t)(0xffffffffu - (uint32_t)(m0 & 0xffffffffu));
            out_scores[row * K + b0] = __uint_as_float((ob & 0x80000000u) ? (ob & 0x7fffffffu) : ~ob);
        }
        if (lane + 32 < n_keep && b1 < K) {
            const uint32_t ob = (uint32_t)(m1 >> 32);
            out_ids[row * K + b1] = (int32_t)(0xffffffffu - (uint32_t)(m1 & 0xffffffffu));
            out_scores[row * K + b1] = __uint_as_float((ob & 0x80000000u) ? (ob & 0x7fffffffu) : ~ob);
        }
        filled = n_keep < K ? n_keep : K;
    } else {
        prev = ~0ull;
        for (int r = 0; r < K; ++r) {
            best = 0ull;
            for (int j = lane; j < n_keep; j += 32) {
                const unsigned long long k = keys[warp][j];
                if (k < prev && k > best) best = k;
            }
            best = warp_max_u64(best);
            if (best == 0ull) break;
            prev = best;
            if (lane == 0) {
                const uint32_t ob = (uint32_t)(best >> 32);
                out_ids[row * K + r] = (int32_t)(0xffffffffu - (uint32_t)(best & 0xffffffffu));
                out_scores[row * K + r] = __uint_as_float((ob & 0x80000000u) ? (ob & 0x7fffffffu) : ~ob);
            }
            ++filled;
        }
    }
    rs_fill_masked(train_indptr, train_indices, u, row, K, filled, lane, 32, out_ids, out_scores);
}

// ------------------------------------------------------------------------------------------ 4. brute force
constexpr int BF_THREADS = 256;

// Block per user: every item scored in fp32 in the canonical order into a scratch row, training items
// overwritten with -10e8, then K rounds of block-wide arg-max under the previous winner.
// only_overflow != 0: process only rows flagged by the tensor path.
__global__ void __launch_bounds__(BF_THREADS) eval_brute_kernel(const float *__restrict__ user_emb,
                                                                const float *__restrict__ item_emb, int D, int n_items,
                                                                const int32_t *__restrict__ test_users,
                                                                const int64_t *__restrict__ train_indptr,
                                                                const int32_t *__restrict__ train_indices,
                                                                const int32_t *__restrict__ overflow, int only_overflow,
                                                                int64_t n_pad, int n_test, int K, float *__restrict__ scratch,
                                                                int32_t *__restrict__ out_ids, float *__restrict__ out_scores,
                                                                unsigned long long *__restrict__ stats) {
    __shared__ float u_sm[128];
    __shared__ unsigned long long red[BF_THREADS / 32];
    __shared__ unsigned long long winner;
    float *srow = scratch + (int64_t)blockIdx.x * n_items;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n_rows = only_overflow ? overflow[n_pad] : n_test;
    for (int q = blockIdx.x; q < n_rows; q += gridDim.x) {
        const int row = only_overflow ? overflow[n_pad + 2 + q] : q;
        const int32_t u = test_users[row];
        __syncthreads();
        for (int k = threadIdx.x; k < D; k += BF_THREADS) u_sm[k] = user_emb[(int64_t)u * D + k];
        __syncthreads();
        for (int i = threadIdx.x; i < n_items; i += BF_THREADS) srow[i] = exact_score(u_sm, item_emb + (int64_t)i * D, D);
        __syncthreads();
        for (int64_t q = train_indptr[u] + threadIdx.x; q < train_indptr[u + 1]; q += BF_THREADS) {
            const int it = train_indices[q];
            if (it >= 0 && it < n_items) srow[it] = EV_MASK_SCORE;
        }
        __syncthreads();
        if (threadIdx.x == 0 && stats && only_overflow) atomicAdd(stats + 2, 1ull);
        unsigned long long prev = ~0ull;
        for (int r = 0; r < K; ++r) {
            unsigned long long best = 0ull;
            for (int i = threadIdx.x; i < n_items; i += BF_THREADS) {
                const unsigned long long k = rank_key(srow[i], i);
                if (k < prev && k > best) best = k;
            }
            best = warp_max_u64(best);
            if (lane == 0) red[warp] = best;
            __syncthreads();
            if (threadIdx.x == 0) {
                unsigned long long b = 0ull;
                for (int w = 0; w < BF_THREADS / 32; ++w) b = red[w] > b ? red[w] : b;
                winner = b;
                if (b != 0ull) {
                    const int id = (int32_t)(0xffffffffu - (uint32_t)(b & 0xffffffffu));
                    out_ids[(int64_t)row * K + r] = id;
                    out_scores[(int64_t)row * K + r] = srow[id];
                } else {
                    out_ids[(int64_t)row * K + r] = -1;
                    out_scores[(int64_t)row * K + r] = EV_MASK_SCORE;
                }
            }
            __syncthreads();
            prev = winner;
            if (prev == 0ull) prev = 1ull;  // nothing left: later rounds find nothing either
        }
    }
}

// ------------------------------------------------------------------------------------------ 5. refquirk
// find_k_largest (util/algorithm.py:143-173) seeds its list with candidates[0:K] sorted by score and then
// visits EVERY candidate again, including those first K (SURVEY.md F9).  Its result is the first K entries
// of the stable merge of  A = items 0..K-1 sorted (score desc, id asc)  and  B = the exact top-K,
// with A's entries first on equal scores.  A group of TPU threads per user, UPB users per block, K <= KMAX: one warp per
// user for K <= 64, one block per user for long lists.
template <int KMAX, int UPB, int TPU>
__global__ void __launch_bounds__(UPB * TPU) eval_refquirk_kernel(const float *__restrict__ user_emb,
                                                                  const float *__restrict__ item_emb, int D,
                                                                  const int32_t *__restrict__ test_users,
                                                                  const int64_t *__restrict__ train_indptr,
                                                                  const int32_t *__restrict__ train_indices, int n_test, int K,
                                                                  int32_t *__restrict__ out_ids, float *__restrict__ out_scores) {
    static_assert(TPU == 32 || UPB == 1, "a user's group is a warp or the whole block");
    __shared__ float u_sm[UPB][128];
    __shared__ float a_s[UPB][KMAX], b_s[UPB][KMAX];
    __shared__ int b_id[UPB][KMAX];
    const int warp = threadIdx.x / TPU, lane = threadIdx.x % TPU;  // warp = the user's group, lane = thread within it
    const int64_t row = (int64_t)blockIdx.x * UPB + warp;
    if (row >= n_test) return;
    const int32_t u = test_users[row];
    for (int k = lane; k < D; k += TPU) u_sm[warp][k] = user_emb[(int64_t)u * D + k];
    if (TPU == 32) __syncwarp();
    else __syncthreads();
    const int64_t t0 = train_indptr[u], t1 = train_indptr[u + 1];
    for (int j = lane; j < K; j += TPU) {
        float s = exact_score(u_sm[warp], item_emb + (int64_t)j * D, D);
        if (is_train_item(train_indices, t0, t1, j)) s = EV_MASK_SCORE;
        a_s[warp][j] = s;
        b_s[warp][j] = out_scores[row * K + j];
        b_id[warp][j] = out_ids[row * K + j];
    }
    if (TPU == 32) __syncwarp();
    else __syncthreads();
    for (int j = lane; j < K; j += TPU) {
        // position of A_j in the merge: A entries ahead of it + B entries with a strictly larger score
        const float s = a_s[warp][j];
        int pos = 0;
        for (int l = 0; l < K; ++l) {
            const float t = a_s[warp][l];
            pos += (t > s) || (t == s && l < j);
            pos += b_s[warp][l] > s;
        }
        if (pos < K) {
            out_ids[row * K + pos] = j;
            out_scores[row * K + pos] = s;
        }
        // position of B_j: B entries ahead of it (B is already sorted) + A entries with score >= its score
        const float sb = b_s[warp][j];
        int pb = j;
        for (int l = 0; l < K; ++l) pb += a_s[warp][l] >= sb;
        if (pb < K) {
            out_ids[row * K + pb] = b_id[warp][j];
            out_scores[row * K + pb] = sb;
        }
    }
}

// ------------------------------------------------------------------------------------------ host side
struct EvalPlan {
    int64_t n_test_pad, n_items_pad;
    int n_tiles, cap, n_brute_blocks, n_mblk;
    int n_seg, seg_tiles, seg_pitch, s_sub, s_sub_tiles;  // sample pass: segment y scores tiles [y * seg_pitch, + seg_tiles) in s_sub sub-ranges
    int stride;                                           // the sample pass scores 1 / stride of the catalogue
    int f_sub, f_sub_tiles;                               // filter pass: all tiles in f_sub sub-ranges
    size_t off_ap, off_bp, off_slack, off_maxnorm, off_bucket, bucket_bytes, off_thr, off_cand, off_cnt, off_overflow, off_scratch, total;
    bool tensor;
    bool pool;  // long lists (EV_LIST_K < K <= EV_MAX_K): one candidate pool of `cap` slots per user
};

static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

constexpr int EV_PLAN_SMS = 148;         // the plan (and with it the workspace size) must not depend on the device it runs on
constexpr int EV_CELLS_PER_SM = 16;      // cells per CTA of the persistent grid: a CTA's share differs from the mean by <= 1 / 16

static EvalPlan make_plan(int64_t n_test, int64_t n_items, int D, int K, int engine) {
    EvalPlan p;
    memset(&p, 0, sizeof(p));
    p.tensor = engine != 1 && D == EV_D && K <= EV_MAX_K && n_test > 0;
    p.pool = p.tensor && K > EV_LIST_K;
    p.n_test_pad = ceil_div(n_test > 0 ? n_test : 1, EV_BM) * EV_BM;
    p.n_items_pad = ceil_div(n_items > 0 ? n_items : 1, EV_BN) * EV_BN;
    p.n_tiles = (int)(p.n_items_pad / EV_BN);

    p.n_mblk = (int)(p.n_test_pad / EV_BM);
    const int64_t want_ranges = ceil_div((int64_t)EV_CELLS_PER_SM * EV_PLAN_SMS, p.n_mblk);  // sub-ranges per user block for ~16 cells per SM
    // filter pass: the whole catalogue in sub-ranges of at least 8 tiles
    {
        int64_t sub = want_ranges;
        const int64_t max_sub = p.n_tiles / 8 > 0 ? p.n_tiles / 8 : 1;
        if (sub > max_sub) sub = max_sub;
        if (sub > 24) sub = 24;
        if (sub < 1) sub = 1;
        p.f_sub_tiles = (int)ceil_div(p.n_tiles, sub);
        p.f_sub = (int)ceil_div(p.n_tiles, p.f_sub_tiles);
        // candidate slots: every (sub-range, column half, user) owns `cap` of them.  A user keeps ~4 K candidates in all (the
        // threshold comes from a 1 / 4 sample), but NOT spread evenly: with ids handed out in order of first appearance the
        // popular items share the first tiles, so a single list must be able to take the user's whole set (4 K and some).  A
        // list that still overflows sends its user to the exact brute-force kernel.  parts * n_test_pad <= ~1.2 M lists by
        // construction (EV_CELLS_PER_SM), i.e. < 1 GB of slots at K = 20.
        int cap = (4 * K + 7) / 8 * 8;
        if (cap < 64) cap = 64;
        if (cap > 512) cap = 512;
        // long lists: slots scale with the users, not with the lists.  A user keeps ~4.5 - 5.5 K candidates (K-th of 2 K bucket
        // maxima from the 1 / 4 sample), so its pool holds EV_POOL_PER_K * K; at most the f_sub * 2 * 256 slots a user owns at
        // K = 64, so that no long list needs more workspace than K = 64 at the same shape.  8 K <= 2048 keys: one block of
        // eval_rescore_kernel sorts the whole pool in 16 KB of shared memory.
        if (p.pool) {
            cap = EV_POOL_PER_K * K;
            if (cap > p.f_sub * EV_CSPLIT * 256) cap = p.f_sub * EV_CSPLIT * 256;
        }
        p.cap = cap;
    }
    // sample pass: n_seg contiguous segments spread evenly over the catalogue, together 1 / stride of it;
    // at least 4 segments (128 buckets >= K), each cut into sub-ranges of at least 4 tiles for the scheduler
    int seg = (int)ceil_div(2 * EV_PLAN_SMS, p.n_mblk);
    if (seg < 4) seg = 4;
    if (seg > 8) seg = 8;  // eval_tau_kernel holds n_seg * sub * EV_CSPLIT <= 16 keys per lane
    // long lists: 8 segments of one sub-range each, so all 16 sets of 32 buckets exist (512 bucket maxima >= 2 K) whatever the
    // number of users (5 - 7 segments would leave 10 - 14 sets); the same number of cells as 4 segments of 2 sub-ranges
    if (p.pool) seg = 8;
    if (seg > p.n_tiles) seg = p.n_tiles;
    p.seg_pitch = p.n_tiles / seg;
    p.n_seg = seg;
    // long lists whose pool is capped below 8 K (many users: few sub-ranges) sample a larger share.  With N = 512 bucket maxima a
    // user keeps about -N ln(1 - K / N) * stride <= 1.39 K * stride candidates (N >= 2 K), and a pool that fills up costs the
    // brute-force kernel.  A catalogue of fewer than 8 tiles has fewer sets, but then seg_pitch = 1 and the sample is all of it.
    p.stride = EV_SAMPLE_STRIDE;
    if (p.pool)
        while (p.stride > 1 && p.cap < 2 * K * p.stride) p.stride /= 2;
    p.seg_tiles = (int)ceil_div(p.seg_pitch, p.stride);
    {
        int64_t sub = ceil_div(want_ranges, seg);
        const int64_t max_sub = p.seg_tiles / 4 > 0 ? p.seg_tiles / 4 : 1;
        if (sub > max_sub) sub = max_sub;
        if (sub > 8 / seg) sub = 8 / seg;  // every (segment, sub-range, column half) owns 32 buckets; eval_tau_kernel merges <= 16 sets
        if (p.pool) sub = 1;  // long lists: 8 segments x 1 sub-range x 2 column halves = 16 sets
        if (sub < 1) sub = 1;
        p.s_sub_tiles = (int)ceil_div(p.seg_tiles, sub);
        p.s_sub = (int)ceil_div(p.seg_tiles, p.s_sub_tiles);
    }
    p.n_brute_blocks = p.tensor ? 148 : 148 * 4;
    if (p.n_brute_blocks > n_test && n_test > 0) p.n_brute_blocks = (int)n_test;
    size_t o = 0;
    if (p.tensor) {
        p.off_ap = o; o = align_up(o + (size_t)p.n_test_pad * EV_D * 2 * 2, 256);
        p.off_bp = o; o = align_up(o + (size_t)p.n_items_pad * EV_D * 2 * 2, 256);
        p.off_slack = o; o = align_up(o + (size_t)p.n_test_pad * 4, 256);
        p.off_maxnorm = o; o = align_up(o + 256, 256);
        p.bucket_bytes = (size_t)8 * EV_CSPLIT * p.n_test_pad * EV_BUCKETS * 4;
        p.off_bucket = o; o = align_up(o + p.bucket_bytes, 256);
        p.off_thr = o; o = align_up(o + (size_t)p.n_test_pad * 4, 256);
        const size_t lists = p.pool ? (size_t)p.n_test_pad : (size_t)p.f_sub * EV_CSPLIT * p.n_test_pad;
        p.off_cand = o; o = align_up(o + lists * p.cap * 8, 256);
        p.off_cnt = o; o = align_up(o + lists * 4, 256);
    }
    p.off_overflow = o; o = align_up(o + (size_t)(3 * p.n_test_pad + 2) * 4, 256);
    p.off_scratch = o; o = align_up(o + (size_t)p.n_brute_blocks * (size_t)(n_items > 0 ? n_items : 1) * 4, 256);
    p.total = o;
    return p;
}

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-device attribute: set it once for every device this process uses
template <int MODE>
static cudaError_t ensure_scores_smem(size_t smem) {
    static std::atomic<uint64_t> done[2];
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    const uint64_t bit = 1ull << (dev & 63);
    if (dev < 128 && (done[(dev >> 6) & 1].load(std::memory_order_acquire) & bit)) return cudaSuccess;
    e = cudaFuncSetAttribute(eval_scores_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess && dev < 128) done[(dev >> 6) & 1].fetch_or(bit, std::memory_order_release);
    return e;
}

static int device_sm_count() {
    static std::atomic<int> cached[128];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return EV_PLAN_SMS;
    if (dev < 128 && cached[dev].load(std::memory_order_relaxed) > 0) return cached[dev].load(std::memory_order_relaxed);
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = EV_PLAN_SMS;
    if (dev < 128) cached[dev].store(n, std::memory_order_relaxed);
    return n;
}

}  // namespace hgr

extern "C" {

size_t hgr_fullrank_topk_workspace_bytes(int64_t n_test, int64_t n_items, int32_t D, int32_t K, int32_t engine) {
    if (n_test < 0 || n_items <= 0 || K <= 0) return 0;
    return hgr::make_plan(n_test, n_items, D, K, engine).total;
}

int hgr_fullrank_topk_f32(const float *user_emb, int64_t n_users, const float *item_emb, int64_t n_items, int32_t D,
                          const int32_t *test_users, int64_t n_test, const int64_t *train_indptr,
                          const int32_t *train_indices, int32_t K, int32_t mode, int32_t engine, int32_t *out_ids,
                          float *out_scores, uint64_t *stats, void *workspace, size_t workspace_bytes,
                          hgr_stream_t stream) {
    using namespace hgr;
    cudaStream_t st = (cudaStream_t)stream;
    HGR_REQUIRE(n_test >= 0 && n_users > 0 && n_items > 0, "negative or empty dimension");
    HGR_REQUIRE(D == 32 || D == 64 || D == 128, "D = %d unsupported (32, 64 or 128)", D);
    HGR_REQUIRE(K >= 1 && K <= n_items, "K = %d must be in [1, n_items = %lld]", K, (long long)n_items);
    HGR_REQUIRE(mode == 0 || mode == 1, "mode %d unknown (0 exact, 1 refquirk)", mode);
    HGR_REQUIRE(engine >= 0 && engine <= 2, "engine %d unknown (0 auto, 1 simt, 2 tensor)", engine);
    HGR_REQUIRE(mode == 0 || K <= EV_MAX_K, "refquirk mode supports K <= 256, got %d", K);
    HGR_REQUIRE(n_items < (int64_t)0x7fffff00 && n_test < (int64_t)0x7fffff00, "dimension does not fit int32");
    if (n_test == 0) return HGR_OK;
    HGR_REQUIRE(user_emb && item_emb && test_users && train_indptr && out_ids && out_scores, "NULL argument");
    HGR_REQUIRE(aligned16(user_emb) && aligned16(item_emb), "embedding tables must be 16-byte aligned");
    const EvalPlan p = make_plan(n_test, n_items, D, K, engine);
    HGR_REQUIRE(engine != 2 || p.tensor, "tensor engine needs D == 64 and K <= 256");
    if (workspace == nullptr || workspace_bytes < p.total)
        return set_error(HGR_ERR_WORKSPACE, "fullrank_topk workspace: need %zu bytes, got %zu", p.total, workspace_bytes);
    HGR_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255u) == 0, "workspace must be 256-byte aligned");
    uint8_t *ws = static_cast<uint8_t *>(workspace);
    int32_t *overflow = reinterpret_cast<int32_t *>(ws + p.off_overflow);
    float *scratch = reinterpret_cast<float *>(ws + p.off_scratch);
    unsigned long long *st64 = reinterpret_cast<unsigned long long *>(stats);
    HGR_CUDA_OK(cudaMemsetAsync(overflow, 0, (size_t)(p.n_test_pad + 2) * 4, st));

    if (p.tensor) {
        __nv_bfloat16 *Ap = reinterpret_cast<__nv_bfloat16 *>(ws + p.off_ap);
        __nv_bfloat16 *Bp = reinterpret_cast<__nv_bfloat16 *>(ws + p.off_bp);
        float *slack = reinterpret_cast<float *>(ws + p.off_slack);
        float *thr = reinterpret_cast<float *>(ws + p.off_thr);
        unsigned int *maxnorm = reinterpret_cast<unsigned int *>(ws + p.off_maxnorm);
        HGR_CUDA_OK(cudaMemsetAsync(maxnorm, 0, 4, st));
        eval_pack_kernel<<<(unsigned)ceil_div(p.n_items_pad * 8, 256), 256, 0, st>>>(item_emb, nullptr, n_items, p.n_items_pad,
                                                                                    n_items, Bp, nullptr, maxnorm);
        HGR_LAUNCH_OK("eval_pack_kernel(items)");
        eval_pack_kernel<<<(unsigned)ceil_div(p.n_test_pad * 8, 256), 256, 0, st>>>(user_emb, test_users, n_test, p.n_test_pad,
                                                                                   n_users, Ap, slack, nullptr);
        HGR_LAUNCH_OK("eval_pack_kernel(users)");
        eval_slack_kernel<<<(unsigned)ceil_div(p.n_test_pad, 256), 256, 0, st>>>(slack, p.n_test_pad, maxnorm);
        HGR_LAUNCH_OK("eval_slack_kernel");

        EvalParams P;
        memset(&P, 0, sizeof(P));
        P.Ap = Ap;
        P.Bp = Bp;
        P.a_term_stride = p.n_test_pad * EV_D * 2;
        P.b_term_stride = p.n_items_pad * EV_D * 2;
        P.test_users = test_users;
        P.train_indptr = train_indptr;
        P.train_indices = train_indices;
        P.bucket_max = reinterpret_cast<float *>(ws + p.off_bucket);
        P.thr = thr;
        P.cand = reinterpret_cast<float2 *>(ws + p.off_cand);
        P.cand_cnt = reinterpret_cast<int32_t *>(ws + p.off_cnt);
        P.overflow = overflow;
        P.n_test = (int32_t)n_test;
        P.n_items = (int32_t)n_items;
        P.n_tiles = p.n_tiles;
        P.n_mblk = p.n_mblk;
        P.cap = p.cap;
        const size_t smem = 1024 + (size_t)EvalSmem::END;
        HGR_CUDA_OK(ensure_scores_smem<EV_SAMPLE>(smem));
        HGR_CUDA_OK(p.pool ? ensure_scores_smem<EV_FILTER_POOL>(smem) : ensure_scores_smem<EV_FILTER>(smem));
        // dead rows and empty cells write nothing; the pools' append counters start at 0
        HGR_CUDA_OK(cudaMemsetAsync(P.cand_cnt, 0, (p.pool ? (size_t)1 : (size_t)p.f_sub * EV_CSPLIT) * p.n_test_pad * 4, st));
        const int n_sm = device_sm_count();
        // persistent grids: one CTA per SM walks its share of the cells (EvalParams)
        P.n_seg = p.n_seg;
        P.seg_pitch = p.seg_pitch;
        P.seg_tiles = p.seg_tiles;
        P.sub = p.s_sub;
        P.sub_tiles = p.s_sub_tiles;
        int64_t cells = (int64_t)p.n_mblk * P.n_seg * P.sub;
        eval_scores_kernel<EV_SAMPLE><<<(unsigned)(cells < n_sm ? cells : n_sm), EV_THREADS, smem, st>>>(P);
        HGR_LAUNCH_OK("eval_scores_kernel<sample>");
        if (p.pool)
            eval_tau_kernel<true><<<(unsigned)ceil_div(n_test, 4), 128, 0, st>>>(P.bucket_max, p.n_seg * p.s_sub * EV_CSPLIT, p.n_test_pad, (int)n_test, K, slack, thr);
        else
            eval_tau_kernel<false><<<(unsigned)ceil_div(n_test, 4), 128, 0, st>>>(P.bucket_max, p.n_seg * p.s_sub * EV_CSPLIT, p.n_test_pad, (int)n_test, K, slack, thr);
        HGR_LAUNCH_OK("eval_tau_kernel");
        P.n_seg = 1;
        P.seg_pitch = 0;
        P.seg_tiles = p.n_tiles;
        P.sub = p.f_sub;
        P.sub_tiles = p.f_sub_tiles;
        cells = (int64_t)p.n_mblk * P.sub;
        if (p.pool) {
            eval_scores_kernel<EV_FILTER_POOL><<<(unsigned)(cells < n_sm ? cells : n_sm), EV_THREADS, smem, st>>>(P);
            HGR_LAUNCH_OK("eval_scores_kernel<filter_pool>");
            int pool_pow = 1;
            while (pool_pow < p.cap) pool_pow <<= 1;
            eval_rescore_kernel<RS_POOL_MAX, -1, 4, RS_POOL_WARPS><<<(unsigned)n_test, RS_POOL_WARPS * 32, (size_t)pool_pow * 8, st>>>(
                user_emb, item_emb, D, test_users, train_indptr, train_indices, P.cand, P.cand_cnt, slack, overflow, 1,
                p.n_test_pad, p.cap, (int)n_test, K, out_ids, out_scores, st64);
            HGR_LAUNCH_OK("eval_rescore_kernel<pool>");
        } else {
            eval_scores_kernel<EV_FILTER><<<(unsigned)(cells < n_sm ? cells : n_sm), EV_THREADS, smem, st>>>(P);
            HGR_LAUNCH_OK("eval_scores_kernel<filter>");
            eval_rescore_kernel<256, -1, 8><<<(unsigned)ceil_div(n_test, RS_WARPS), RS_WARPS * 32, 0, st>>>(
                user_emb, item_emb, D, test_users, train_indptr, train_indices, P.cand, P.cand_cnt, slack, overflow,
                p.f_sub * EV_CSPLIT, p.n_test_pad, p.cap, (int)n_test, K, out_ids, out_scores, st64);
            HGR_LAUNCH_OK("eval_rescore_kernel<256>");
            eval_rescore_kernel<RS_CAP, 256, 1><<<(unsigned)ceil_div(n_test, RS_WARPS), RS_WARPS * 32, 0, st>>>(
                user_emb, item_emb, D, test_users, train_indptr, train_indices, P.cand, P.cand_cnt, slack, overflow,
                p.f_sub * EV_CSPLIT, p.n_test_pad, p.cap, (int)n_test, K, out_ids, out_scores, st64);
            HGR_LAUNCH_OK("eval_rescore_kernel<1024>");
        }
    }
    eval_brute_kernel<<<(unsigned)p.n_brute_blocks, BF_THREADS, 0, st>>>(user_emb, item_emb, D, (int)n_items, test_users,
                                                                        train_indptr, train_indices, overflow, p.tensor ? 1 : 0,
                                                                        p.n_test_pad, (int)n_test, K, scratch, out_ids, out_scores, st64);
    HGR_LAUNCH_OK("eval_brute_kernel");
    if (mode == 1 && K <= EV_LIST_K) {
        eval_refquirk_kernel<EV_LIST_K, 4, 32><<<(unsigned)ceil_div(n_test, 4), 128, 0, st>>>(user_emb, item_emb, D, test_users, train_indptr,
                                                                                              train_indices, (int)n_test, K, out_ids, out_scores);
        HGR_LAUNCH_OK("eval_refquirk_kernel");
    } else if (mode == 1) {
        eval_refquirk_kernel<EV_MAX_K, 1, EV_MAX_K><<<(unsigned)n_test, EV_MAX_K, 0, st>>>(user_emb, item_emb, D, test_users, train_indptr,
                                                                                           train_indices, (int)n_test, K, out_ids, out_scores);
        HGR_LAUNCH_OK("eval_refquirk_kernel<long>");
    }
    return HGR_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------ ranking metrics
// Per-user pieces of util/evaluation.py (Metric.hits :9-15, Metric.NDCG :85-97) from the [n_test, K] id matrix:
//   hits[r][q] = | set(truth of r) ∩ set(ids[r][:N_q]) |      (a duplicated recommendation counts once)
//   dcg[r][q]  = sum over positions p < N_q with ids[r][p] in truth of disc[p]   (duplicates count every time, in
//                position order, in double: the same additions as the python loop)
// disc[p] = 1.0 / math.log(p + 2, 2) is passed in by the host so that the doubles are python's own.
// One thread per user; truth rows sorted ascending (binary search); the sums over users stay on the host, in the
// reference's order, so the rounded metric strings are identical.
namespace hgr {
__global__ void __launch_bounds__(128) rank_metrics_kernel(const int32_t *__restrict__ ids, int n_test, int K,
                                                           const int64_t *__restrict__ truth_indptr,
                                                           const int32_t *__restrict__ truth_items, const int32_t *__restrict__ top_n,
                                                           int n_top, const double *__restrict__ disc, int32_t *__restrict__ hits,
                                                           double *__restrict__ dcg) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_test) return;
    const int64_t t0 = truth_indptr[r], t1 = truth_indptr[r + 1];
    const int32_t *row = ids + (int64_t)r * K;
    int h = 0;
    double d = 0.0;
    int q = 0;
    for (int p = 0; p < K && q < n_top; ++p) {
        const int id = row[p];
        if (id >= 0 && is_train_item(truth_items, t0, t1, id)) {
            d += disc[p];
            bool first = true;
            for (int e = 0; e < p; ++e) first = first && row[e] != id;
            h += first;
        }
        while (q < n_top && p + 1 == top_n[q]) {  // top_n ascending
            hits[(int64_t)r * n_top + q] = h;
            dcg[(int64_t)r * n_top + q] = d;
            ++q;
        }
    }
    for (; q < n_top; ++q) {  // N_q > K: the list is shorter than N
        hits[(int64_t)r * n_top + q] = h;
        dcg[(int64_t)r * n_top + q] = d;
    }
}
}  // namespace hgr

// The sums over users of util/evaluation.py (Metric.hit_ratio :18-30, precision :45-48, recall :50-53, NDCG :85-97) in the
// reference's own ORDER of floating-point additions, on the device: 256 threads form the per-user terms of a chunk of users
// in parallel (hits / n_truth and dcg / idcg are correctly rounded double divisions, as in python), then ONE thread per sum
// adds the chunk's terms sequentially in user order.  `compensated`: python >= 3.12's builtin sum() (Neumaier) for the
// recall list; the NDCG loop is a plain `+=` in every version.  262 144 users: ~3 ms instead of 0.2 s of python loops.
namespace hgr {
__global__ void __launch_bounds__(256) rank_metric_sums_kernel(const int32_t *__restrict__ hits, const double *__restrict__ dcg,
                                                               const int64_t *__restrict__ truth_indptr, int n_test, int n_top,
                                                               const int32_t *__restrict__ top_n, const double *__restrict__ idcg_tab,
                                                               int idcg_len, int compensated, long long *__restrict__ hit_sum,
                                                               double *__restrict__ recall_sum, double *__restrict__ ndcg_sum) {
    __shared__ double s_rec[256], s_ndcg[256];
    __shared__ int s_hit[256];
    const int t = threadIdx.x;
    for (int q = 0; q < n_top; ++q) {
        const int N = top_n[q];
        double rs = 0.0, rc = 0.0, ns = 0.0;
        long long hs = 0;
        for (int base = 0; base < n_test; base += 256) {
            const int r = base + t;
            if (r < n_test) {
                const long long nt = truth_indptr[r + 1] - truth_indptr[r];
                const int h = hits[(int64_t)r * n_top + q];
                s_hit[t] = h;
                s_rec[t] = nt > 0 ? (double)h / (double)nt : 0.0;
                long long k = nt < N ? nt : N;
                if (k >= idcg_len) k = idcg_len - 1;
                s_ndcg[t] = k > 0 ? dcg[(int64_t)r * n_top + q] / idcg_tab[k] : 0.0;
            }
            __syncthreads();
            const int cnt = n_test - base < 256 ? n_test - base : 256;
            if (t == 0) {
                if (compensated) {
                    for (int j = 0; j < cnt; ++j) {
                        const double x = s_rec[j];
                        const double y = rs + x;
                        if (fabs(rs) >= fabs(x)) rc += (rs - y) + x;
                        else rc += (x - y) + rs;
                        rs = y;
                    }
                } else {
                    for (int j = 0; j < cnt; ++j) rs += s_rec[j];
                }
            } else if (t == 32) {
                for (int j = 0; j < cnt; ++j) ns += s_ndcg[j];
            } else if (t == 64) {
                for (int j = 0; j < cnt; ++j) hs += s_hit[j];
            }
            __syncthreads();
        }
        if (t == 0) recall_sum[q] = (compensated && rc != 0.0 && isfinite(rc)) ? rs + rc : rs;
        if (t == 32) ndcg_sum[q] = ns;
        if (t == 64) hit_sum[q] = hs;
    }
}
}  // namespace hgr

extern "C" int hgr_rank_metric_sums(const int32_t *hits, const double *dcg, const int64_t *truth_indptr, int64_t n_test, int32_t n_top,
                                    const int32_t *top_n, const double *idcg_tab, int32_t idcg_len, int32_t compensated,
                                    int64_t *hit_sum, double *recall_sum, double *ndcg_sum, hgr_stream_t stream) {
    using namespace hgr;
    HGR_REQUIRE(n_test >= 0 && n_test < (int64_t)0x7fffff00 && n_top >= 1 && n_top <= 16 && idcg_len >= 1, "bad n_test / n_top / idcg_len");
    HGR_REQUIRE(hits && dcg && truth_indptr && top_n && idcg_tab && hit_sum && recall_sum && ndcg_sum, "NULL argument");
    rank_metric_sums_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(hits, dcg, truth_indptr, (int)n_test, n_top, top_n, idcg_tab, idcg_len,
                                                              compensated, reinterpret_cast<long long *>(hit_sum), recall_sum, ndcg_sum);
    HGR_LAUNCH_OK("rank_metric_sums_kernel");
    return HGR_OK;
}

extern "C" int hgr_rank_metrics(const int32_t *ids, int64_t n_test, int32_t K, const int64_t *truth_indptr, const int32_t *truth_items,
                                const int32_t *top_n, int32_t n_top, const double *disc, int32_t *hits, double *dcg,
                                hgr_stream_t stream) {
    using namespace hgr;
    HGR_REQUIRE(n_test >= 0 && K >= 1 && n_top >= 1 && n_top <= 16, "bad n_test / K / n_top");
    if (n_test == 0) return HGR_OK;
    HGR_REQUIRE(ids && truth_indptr && top_n && disc && hits && dcg, "NULL argument");
    rank_metrics_kernel<<<(unsigned)ceil_div(n_test, 128), 128, 0, (cudaStream_t)stream>>>(ids, (int)n_test, K, truth_indptr, truth_items,
                                                                                         top_n, n_top, disc, hits, dcg);
    HGR_LAUNCH_OK("rank_metrics_kernel");
    return HGR_OK;
}
