// Sparse embedding propagation Y = epilogue(A . X) for sm_100a.
//
// Replaces torch.sparse.mm(adj, X) at model/graph/LightGCN.py:133, HCCF.py:199,
// HGNN_HD3.py:549-553 of the reference, plus the elementwise / LayerNorm / residual / readout
// kernels torch launches after it (SURVEY.md K1-K4).
//
// Mapping.  One embedding row is D fp32 = D/4 128-bit words, so a "row group" of LPR = D/4 lanes
// owns one output row and every gathered X row is a single fully coalesced 128-bit-per-lane load
// (D = 64: a half warp reads one 256-byte row, a warp works on two output rows).  The group walks
// its nonzeros in stored order and keeps ONE accumulator chain per feature, so a row that is not
// split is accumulated with exactly the fused multiply-add sequence of the CPU oracle
// (oracle/hgr_oracle.c) and is bit-identical to it.  Memory-level parallelism comes from keeping
// the gathers of the next nonzeros in flight (cp.async into a shared-memory ring) while the
// current ones are accumulated, and from prefetching the next (column, value) batches -- not from
// splitting the sum.
//
// Power-law rows.  Rows longer than plan.chunk_nnz are cut into chunks of chunk_nnz nonzeros; a
// chunk is accumulated by one group into a partial row, and a second kernel adds the partials of a
// row in chunk order and runs the epilogue.  No atomics: results are reproducible run to run.
#include <string.h>

#include "hgr_internal.cuh"

namespace hgr {

constexpr int kThreads = 256;
constexpr int kUnroll = 8;  // partial-row reduce kernel
constexpr int kGroupReduceMax = 64;  // a split row with at most this many chunks is summed by one row group
// Gather ring of 2 x kRingHalf embedding rows per thread, kMinBlocks resident blocks per SM.  Measured on B200
// (profiles/spmm_variants_r1.md): resident warps beat deeper gather batches, staging the gathered rows through shared
// memory with cp.async beats register loads by ~15 %, and 5 blocks leave 48 registers per thread, so the 2 x 4 ring
// compiles without the spills it has under the 40-register cap of 6 blocks (+9 % on both shapes).
constexpr int kRingHalf = 4;
constexpr int kMinBlocks = 5;
static_assert(2 * kRingHalf * kThreads * sizeof(float4) <= 48 * 1024,
              "the gather ring must fit the 48 KB of dynamic shared memory a launch gets without cudaFuncSetAttribute");

// The gather: every lane copies ITS 16 bytes of the next HB embedding rows straight into a per-thread ring in shared
// memory (LDGSTS, L1 bypass) and consumes them in order, so the number of row gathers in flight is bounded by shared
// memory (2 x HB rows per row group) instead of by what the load/store unit tracks for register loads.
__device__ __forceinline__ void cp_async16(void *smem, const void *gmem) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

// Lane gl of a row group holds (column, value) of nonzero `base + gl` of the current batch of LPR nonzeros and of the
// next one (coalesced, prefetched); the embedding rows of sub-batch q + 1 (HB nonzeros) are in flight into one half of
// the ring while sub-batch q is consumed from the other half.
template <int LPR, int HB>
__device__ __forceinline__ float4 gather_accumulate_async(const int32_t *__restrict__ idx, const float *__restrict__ val,
                                                          const float4 *__restrict__ X4, int64_t s, int64_t e, int gl,
                                                          unsigned gmask, float4 *__restrict__ ring /* stride kThreads */) {
    static_assert(LPR % HB == 0, "sub-batch must divide the batch");
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (s >= e) return acc;
    int c = 0, cn = 0;
    float v = 0.f, vn = 0.f;
    if (s + gl < e) {
        c = ld_stream_i32(idx + s + gl);
        v = ld_stream_f32(val + s + gl);
    }
    if (s + LPR + gl < e) {
        cn = ld_stream_i32(idx + s + LPR + gl);
        vn = ld_stream_f32(val + s + LPR + gl);
    }
    // sub-batch 0 of the first batch
#pragma unroll
    for (int k = 0; k < HB; ++k) {
        const int cc = __shfl_sync(gmask, c, k, LPR);
        if (s + k < e) cp_async16(ring + k * kThreads, X4 + (int64_t)cc * LPR + gl);
    }
    cp_async_commit();
    int half = 0;
    for (int64_t base = s; base < e; base += LPR) {
        // (column, value) of the batch after next
        int c2 = 0;
        float v2 = 0.f;
        if (base + 2 * LPR + gl < e) {
            c2 = ld_stream_i32(idx + base + 2 * LPR + gl);
            v2 = ld_stream_f32(val + base + 2 * LPR + gl);
        }
#pragma unroll
        for (int q = 0; q < LPR / HB; ++q) {
            const int64_t sub = base + q * HB;  // first nonzero of the sub-batch being consumed
            if (sub >= e) break;
            // issue the next sub-batch (q + 1 of this batch, or 0 of the next batch) into the other half
            const int64_t nsub = sub + HB;
#pragma unroll
            for (int k = 0; k < HB; ++k) {
                const int src = (q + 1 < LPR / HB) ? (q + 1) * HB + k : k;
                const int cc = __shfl_sync(gmask, (q + 1 < LPR / HB) ? c : cn, src, LPR);
                if (nsub + k < e) cp_async16(ring + ((half ^ 1) * HB + k) * kThreads, X4 + (int64_t)cc * LPR + gl);
            }
            cp_async_commit();
            cp_async_wait<1>();  // everything but the group just committed has landed: sub-batch q is in `half`
#pragma unroll
            for (int k = 0; k < HB; ++k) {
                const float vv = __shfl_sync(gmask, v, q * HB + k, LPR);
                if (sub + k < e) {
                    const float4 x = ring[(half * HB + k) * kThreads];
                    acc.x = fmaf(vv, x.x, acc.x);
                    acc.y = fmaf(vv, x.y, acc.y);
                    acc.z = fmaf(vv, x.z, acc.z);
                    acc.w = fmaf(vv, x.w, acc.w);
                }
            }
            half ^= 1;
        }
        c = cn;
        v = vn;
        cn = c2;
        vn = v2;
    }
    cp_async_wait<0>();
    return acc;
}

__device__ __forceinline__ float leaky(float x, float slope) { return x > 0.f ? x : x * slope; }

template <int LPR>
__device__ __forceinline__ void finish_row(float4 acc, int64_t row, int gl, unsigned gmask, const hgr_epilogue_t &ep,
                                           float *__restrict__ Y) {
    constexpr float kInvD = 1.0f / (float)(LPR * 4);
    const int64_t off = row * LPR + gl;
    if (ep.pre) reinterpret_cast<float4 *>(ep.pre)[off] = acc;
    if (ep.use_leaky) {
        acc.x = leaky(acc.x, ep.leaky_slope);
        acc.y = leaky(acc.y, ep.leaky_slope);
        acc.z = leaky(acc.z, ep.leaky_slope);
        acc.w = leaky(acc.w, ep.leaky_slope);
    }
    if (ep.ln_gamma) {
        const float mean = group_sum<LPR>((acc.x + acc.y) + (acc.z + acc.w), gmask) * kInvD;
        const float dx = acc.x - mean, dy = acc.y - mean, dz = acc.z - mean, dw = acc.w - mean;
        const float var = group_sum<LPR>((dx * dx + dy * dy) + (dz * dz + dw * dw), gmask) * kInvD;
        const float rstd = 1.0f / sqrtf(var + ep.ln_eps);
        const float4 g = __ldg(reinterpret_cast<const float4 *>(ep.ln_gamma) + gl);
        const float4 b = __ldg(reinterpret_cast<const float4 *>(ep.ln_beta) + gl);
        acc.x = dx * rstd * g.x + b.x;
        acc.y = dy * rstd * g.y + b.y;
        acc.z = dz * rstd * g.z + b.z;
        acc.w = dw * rstd * g.w + b.w;
    }
    if (ep.residual) {
        const float4 r = ld_stream_f4(reinterpret_cast<const float4 *>(ep.residual) + off);
        acc.x += r.x;
        acc.y += r.y;
        acc.z += r.z;
        acc.w += r.w;
    }
    if (ep.n_addends > 0) {
        float4 s = ld_stream_f4(reinterpret_cast<const float4 *>(ep.addends[0]) + off);
#pragma unroll
        for (int j = 1; j < HGR_MAX_ADDENDS; ++j) {  // constant indices keep ep in param space
            if (j < ep.n_addends) {
                const float4 a = ld_stream_f4(reinterpret_cast<const float4 *>(ep.addends[j]) + off);
                s.x += a.x;
                s.y += a.y;
                s.z += a.z;
                s.w += a.w;
            }
        }
        acc.x += s.x;
        acc.y += s.y;
        acc.z += s.z;
        acc.w += s.w;
    }
    if (ep.n_addends > 0 || ep.scale_always) {
        acc.x *= ep.scale;
        acc.y *= ep.scale;
        acc.z *= ep.scale;
        acc.w *= ep.scale;
    }
    if (Y) reinterpret_cast<float4 *>(Y)[off] = acc;
    if (ep.gather_mc) {
        // fused all-gather through the switch: one multimem store, replicated by NVSwitch into every rank's gathered table
        st_multicast_f4(reinterpret_cast<float4 *>(ep.gather_mc) + (ep.gather_row_offset + row) * LPR + gl, acc);
    } else if (ep.n_gather > 0) {
        // fused all-gather: the same row into the gathered table of every rank (peer-mapped memory; plain 128-bit
        // stores travel over NVLink as posted writes while the block moves on to its next rows)
        const int64_t goff = (ep.gather_row_offset + row) * LPR + gl;
#pragma unroll
        for (int p = 0; p < HGR_MAX_GATHER; ++p)  // constant indices keep ep in param space
            if (p < ep.n_gather) reinterpret_cast<float4 *>(ep.gather_out[p])[goff] = acc;
    }
}


// What a row group works on: entry blockIdx.x * GPB + g of the work list.  Entry w >= 0 is a whole (unsplit) row, w < 0 is
// chunk ~w of the split plan; the host orders the list (rows binned by length so that the two half-warps of a warp and the
// 16 groups of a block retire together, items ordered by the table window they gather from so a window stays in L2).  The
// order only schedules: every row is still accumulated by ONE group in stored order, so no bit of the result depends on it.
struct WorkItem {
    int64_t s, e;    // nonzero range
    int64_t target;  // row (kind 0) or chunk (kind 1); -1: nothing to do
    int kind;
};

template <int GPB>
__device__ __forceinline__ WorkItem resolve_work(const hgr_csr_t &A, int g) {
    WorkItem w;
    w.s = w.e = 0;
    w.target = -1;
    w.kind = 0;
    const int64_t wi = (int64_t)blockIdx.x * GPB + g;
    if (wi >= A.n_work) return w;
    const int id = A.work_order[wi];
    if (id < 0) {
        const int64_t chunk = (int64_t)(~id);
        const int h = A.chunk_owner[chunk];
        const int r = A.heavy_rows[h];
        const int64_t row_end = A.indptr[r + 1];
        if (A.chunk_start) {  // explicit boundaries (window-aligned plan)
            w.s = A.chunk_start[chunk];
            w.e = chunk + 1 < A.heavy_chunk_ptr[h + 1] ? A.chunk_start[chunk + 1] : row_end;
        } else {
            w.s = A.indptr[r] + (chunk - A.heavy_chunk_ptr[h]) * (int64_t)A.chunk_nnz;
            w.e = w.s + A.chunk_nnz < row_end ? w.s + A.chunk_nnz : row_end;
        }
        w.target = chunk;
        w.kind = 1;
        return w;
    }
    w.s = A.indptr[id];
    w.e = A.indptr[id + 1];
    w.target = id;
    return w;
}

template <int LPR, int HB, int MINB>
__global__ void __launch_bounds__(kThreads, MINB) spmm_rows_async_kernel(hgr_csr_t A, const float4 *__restrict__ X4,
                                                                   float *__restrict__ Y, hgr_epilogue_t ep,
                                                                   float4 *__restrict__ partials) {
    extern __shared__ float4 spmm_ring[];  // [2 * HB][kThreads]
    constexpr int GPB = kThreads / LPR;
    const int gl = threadIdx.x % LPR;
    const int g = threadIdx.x / LPR;
    const unsigned gmask = (LPR == 32) ? 0xffffffffu : (((1u << LPR) - 1u) << ((threadIdx.x % 32) / LPR * LPR));
    float4 *ring = spmm_ring + threadIdx.x;
    const WorkItem w = resolve_work<GPB>(A, g);
    if (w.target < 0) return;
    const float4 acc = gather_accumulate_async<LPR, HB>(A.indices, A.values, X4, w.s, w.e, gl, gmask, ring);
    if (w.kind) partials[w.target * LPR + gl] = acc;
    else finish_row<LPR>(acc, w.target, gl, gmask, ep, Y);
}

// Sums the partial rows of the split rows and runs the epilogue.  A block takes GPB consecutive split rows.  Most of them
// have a handful of chunks (a power-law tail cut at chunk_nnz, or one chunk per table window the row crosses): ONE group adds
// those in chunk order, up to kGroupReduceMax chunks.  A row with more chunks is then reduced by the whole block: group g
// adds chunks g, g + GPB, ... in order, group 0 adds the GPB group sums in group order.
// A fixed order either way: deterministic.  The first version launched one block per split row - 22 000 blocks of which
// all but a few hundred used 1/16 of their threads (0.14 ms per propagation).
template <int LPR>
__global__ void __launch_bounds__(kThreads) spmm_heavy_reduce_kernel(hgr_csr_t A, const float4 *__restrict__ partials,
                                                                     float *__restrict__ Y, hgr_epilogue_t ep) {
    constexpr int GPB = kThreads / LPR;
    __shared__ float4 sh[kThreads];
    const int gl = threadIdx.x % LPR;
    const int g = threadIdx.x / LPR;
    const unsigned gmask = (LPR == 32) ? 0xffffffffu : (((1u << LPR) - 1u) << ((threadIdx.x % 32) / LPR * LPR));
    const int h0 = blockIdx.x * GPB;
    const int h_end = h0 + GPB < A.n_heavy_rows ? h0 + GPB : A.n_heavy_rows;
    {
        const int h = h0 + g;
        if (h < h_end) {
            const int64_t c0 = A.heavy_chunk_ptr[h], c1 = A.heavy_chunk_ptr[h + 1];
            if (c1 - c0 <= kGroupReduceMax) {
                float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
                for (int64_t c = c0; c < c1; c += 4) {  // four loads in flight, added in chunk order
                    float4 p[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        if (c + k < c1) p[k] = ld_stream_f4(partials + (c + k) * LPR + gl);
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        if (c + k < c1) {
                            acc.x += p[k].x;
                            acc.y += p[k].y;
                            acc.z += p[k].z;
                            acc.w += p[k].w;
                        }
                }
                finish_row<LPR>(acc, A.heavy_rows[h], gl, gmask, ep, Y);
            }
        }
    }
    for (int h = h0; h < h_end; ++h) {  // block-uniform loop: the rows with more chunks than groups
        const int64_t c0 = A.heavy_chunk_ptr[h], c1 = A.heavy_chunk_ptr[h + 1];
        if (c1 - c0 <= kGroupReduceMax) continue;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int64_t c = c0 + g; c < c1; c += (int64_t)GPB * kUnroll) {
            float4 p[kUnroll];
#pragma unroll
            for (int k = 0; k < kUnroll; ++k)
                if (c + (int64_t)k * GPB < c1) p[k] = ld_stream_f4(partials + (c + (int64_t)k * GPB) * LPR + gl);
#pragma unroll
            for (int k = 0; k < kUnroll; ++k)
                if (c + (int64_t)k * GPB < c1) {
                    acc.x += p[k].x;
                    acc.y += p[k].y;
                    acc.z += p[k].z;
                    acc.w += p[k].w;
                }
        }
        __syncthreads();  // sh is free again
        sh[threadIdx.x] = acc;
        __syncthreads();
        if (g == 0) {
            for (int k = 1; k < GPB; ++k) {
                const float4 q = sh[k * LPR + gl];
                acc.x += q.x;
                acc.y += q.y;
                acc.z += q.z;
                acc.w += q.w;
            }
            finish_row<LPR>(acc, A.heavy_rows[h], gl, gmask, ep, Y);
        }
    }
}

static int check_csr(const hgr_csr_t *A, const char *name) {
    HGR_REQUIRE(A != nullptr, "%s is NULL", name);
    HGR_REQUIRE(A->n_rows >= 0 && A->n_cols >= 0 && A->nnz >= 0, "%s: negative dimension", name);
    HGR_REQUIRE(A->indptr && (A->nnz == 0 || (A->indices && A->values)), "%s: NULL indptr/indices/values", name);
    if (A->n_heavy_rows > 0) {
        HGR_REQUIRE(A->chunk_nnz > 0 && A->n_chunks > 0, "%s: split plan without chunk size", name);
        HGR_REQUIRE(A->heavy_rows && A->heavy_chunk_ptr && A->chunk_owner, "%s: NULL split-plan arrays", name);
    }
    HGR_REQUIRE(A->n_work >= 0 && (A->work_order != nullptr || A->n_work == 0), "%s: n_work = %lld without a work list", name,
                (long long)A->n_work);
    if (A->work_order)
        HGR_REQUIRE(A->n_work <= (int64_t)A->n_rows + A->n_chunks, "%s: work list longer than rows + chunks", name);
    if (A->chunk_start) HGR_REQUIRE(A->n_heavy_rows > 0, "%s: explicit chunk boundaries need a split plan", name);
    return HGR_OK;
}

static int check_epilogue(const hgr_epilogue_t *ep) {
    if (!ep) return HGR_OK;
    HGR_REQUIRE(ep->n_addends >= 0 && ep->n_addends <= HGR_MAX_ADDENDS, "epilogue: n_addends %d out of range", ep->n_addends);
    HGR_REQUIRE((ep->ln_gamma == nullptr) == (ep->ln_beta == nullptr), "epilogue: ln_gamma and ln_beta must come together");
    HGR_REQUIRE(aligned16(ep->ln_gamma) && aligned16(ep->ln_beta) && aligned16(ep->residual) && aligned16(ep->pre),
                "epilogue: operands must be 16-byte aligned");
    for (int j = 0; j < ep->n_addends; ++j)
        HGR_REQUIRE(ep->addends[j] && aligned16(ep->addends[j]), "epilogue: addend %d NULL or misaligned", j);
    HGR_REQUIRE(ep->n_gather >= 0 && ep->n_gather <= HGR_MAX_GATHER, "epilogue: n_gather %d out of range", ep->n_gather);
    for (int j = 0; j < ep->n_gather; ++j)
        HGR_REQUIRE(ep->gather_out[j] && aligned16(ep->gather_out[j]), "epilogue: gather_out %d NULL or misaligned", j);
    HGR_REQUIRE(ep->gather_row_offset >= 0, "epilogue: negative gather_row_offset");
    HGR_REQUIRE(aligned16(ep->gather_mc), "epilogue: gather_mc must be 16-byte aligned");
    return HGR_OK;
}

template <int LPR>
static int launch_spmm(const hgr_csr_t &A, const float *X, float *Y, const hgr_epilogue_t &ep, void *ws, cudaStream_t st) {
    constexpr int GPB = kThreads / LPR;
    float4 *partials = reinterpret_cast<float4 *>(ws);
    const int64_t grid = ceil_div(A.n_work, GPB);
    if (grid == 0) return HGR_OK;
    HGR_REQUIRE(grid < (int64_t)0x7fffffff, "grid too large (%lld blocks)", (long long)grid);
    const size_t smem = (size_t)2 * kRingHalf * kThreads * sizeof(float4);
    spmm_rows_async_kernel<LPR, kRingHalf, kMinBlocks><<<(unsigned)grid, kThreads, smem, st>>>(A, reinterpret_cast<const float4 *>(X), Y,
                                                                                                ep, partials);
    HGR_LAUNCH_OK("spmm_rows_async_kernel");
    if (A.n_heavy_rows > 0) {
        spmm_heavy_reduce_kernel<LPR><<<(unsigned)ceil_div(A.n_heavy_rows, kThreads / LPR), kThreads, 0, st>>>(A, partials, Y, ep);
        HGR_LAUNCH_OK("spmm_heavy_reduce_kernel");
    }
    return HGR_OK;
}

static int spmm_impl(const hgr_csr_t *A, const float *X, float *Y, int32_t D, const hgr_epilogue_t *epi, void *ws,
                     size_t ws_bytes, cudaStream_t st) {
    int rc = check_csr(A, "A");
    if (rc) return rc;
    rc = check_epilogue(epi);
    if (rc) return rc;
    HGR_REQUIRE(D == 32 || D == 64 || D == 128, "D = %d unsupported (32, 64 or 128)", D);
    HGR_REQUIRE(A->n_rows == 0 || (X && (Y || (epi && (epi->n_gather > 0 || epi->gather_mc)))), "X or Y is NULL");
    HGR_REQUIRE(aligned16(X) && aligned16(Y), "X and Y must be 16-byte aligned");
    const size_t need = hgr_spmm_workspace_bytes(A, D);
    if (need > 0 && (ws == nullptr || ws_bytes < need))
        return set_error(HGR_ERR_WORKSPACE, "spmm workspace: need %zu bytes, got %zu", need, ws_bytes);
    HGR_REQUIRE(aligned16(ws), "workspace must be 16-byte aligned");
    HGR_REQUIRE(A->n_rows == 0 || A->work_order, "A: no work list (hgr_csr_t::work_order is required when n_rows > 0)");
    hgr_epilogue_t ep;
    if (epi) ep = *epi;
    else {
        memset(&ep, 0, sizeof(ep));
        ep.scale = 1.f;
    }
    switch (D) {
        case 32: return launch_spmm<8>(*A, X, Y, ep, ws, st);
        case 64: return launch_spmm<16>(*A, X, Y, ep, ws, st);
        default: return launch_spmm<32>(*A, X, Y, ep, ws, st);
    }
}

}  // namespace hgr

extern "C" {

size_t hgr_spmm_workspace_bytes(const hgr_csr_t *A, int32_t D) {
    if (!A || A->n_heavy_rows <= 0) return 0;
    return (size_t)A->n_chunks * (size_t)D * sizeof(float);
}

int hgr_spmm_f32(const hgr_csr_t *A, const float *X, float *Y, int32_t D, const hgr_epilogue_t *epi, void *workspace,
                 size_t workspace_bytes, hgr_stream_t stream) {
    return hgr::spmm_impl(A, X, Y, D, epi, workspace, workspace_bytes, (cudaStream_t)stream);
}

int hgr_hgconv_f32(const hgr_csr_t *A, const hgr_csr_t *At, const float *X, float *tmp, float *Y, int32_t D,
                   const hgr_epilogue_t *epi, void *workspace, size_t workspace_bytes, hgr_stream_t stream) {
    HGR_REQUIRE(A && At, "A or At is NULL");
    HGR_REQUIRE(A->n_cols == At->n_rows, "A is [%d, %d] but At is [%d, %d]", A->n_rows, A->n_cols, At->n_rows, At->n_cols);
    HGR_REQUIRE(tmp != nullptr || At->n_rows == 0, "tmp is NULL");
    int rc = hgr::spmm_impl(At, X, tmp, D, nullptr, workspace, workspace_bytes, (cudaStream_t)stream);
    if (rc) return rc;
    return hgr::spmm_impl(A, tmp, Y, D, epi, workspace, workspace_bytes, (cudaStream_t)stream);
}

int hgr_lightgcn_forward_f32(const hgr_csr_t *A, const float *E0, float *layers, float *out, int32_t n_layers, int32_t D,
                             int32_t sum_readout, void *workspace, size_t workspace_bytes, hgr_stream_t stream) {
    HGR_REQUIRE(A && E0 && out, "A, E0 or out is NULL");
    HGR_REQUIRE(A->n_rows == A->n_cols, "propagation needs a square adjacency, got [%d, %d]", A->n_rows, A->n_cols);
    HGR_REQUIRE(n_layers >= 1 && n_layers <= HGR_MAX_ADDENDS, "n_layers = %d out of range [1, %d]", n_layers, HGR_MAX_ADDENDS);
    HGR_REQUIRE(n_layers == 1 || layers, "layers buffer is NULL");
    const size_t tab = (size_t)A->n_rows * (size_t)D;
    const float *cur = E0;
    for (int k = 1; k < n_layers; ++k) {
        float *nxt = layers + (size_t)(k - 1) * tab;
        int rc = hgr::spmm_impl(A, cur, nxt, D, nullptr, workspace, workspace_bytes, (cudaStream_t)stream);
        if (rc) return rc;
        cur = nxt;
    }
    hgr_epilogue_t ep;
    memset(&ep, 0, sizeof(ep));
    ep.n_addends = n_layers;
    ep.addends[0] = E0;
    for (int k = 1; k < n_layers; ++k) ep.addends[k] = layers + (size_t)(k - 1) * tab;
    ep.scale = sum_readout ? 1.0f : 1.0f / (float)(n_layers + 1);
    return hgr::spmm_impl(A, cur, out, D, &ep, workspace, workspace_bytes, (cudaStream_t)stream);
}

}  // extern "C"
