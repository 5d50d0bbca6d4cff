// Contrastive (SSL) losses fused with their embedding gathers and row normalisation, forward and backward, sm_100a.
//
// Replaces (SURVEY.md K9)
//   contrastLoss(embeds1, embeds2, nodes, temp)    util/loss_torch.py:103-110, called 2 x n_layers times per batch by
//                                                  HCCF.calcLosses (model/graph/HCCF.py:59-68) and HGNN_HD3.py:345-350
//       a_j = normalize(E1[node_j] + 1e-8),  b_j = normalize(E2[node_j] + 1e-8)        (F.normalize: x / max(||x||, 1e-12))
//       loss = -mean_j log( exp(a_j.b_j / T) / (sum_k exp(a_j.b_k / T) + 1e-8) )
//   InfoNCE(view1, view2, temperature, b_cos)      util/loss_torch.py:32-40, called by SGL.cal_cl_loss (model/graph/SGL.py:167-180)
//       loss = -mean_j log( exp(a_j.b_j / T) / sum_k exp(a_j.b_k / T) + 10e-6 )
// The reference normalises the WHOLE tables (two passes over N x D), materialises the [M, M] logits, and runs
// ~10 kernels; here only the M picked rows are touched and the logits live in registers / shared memory:
//   ssl_prepare_kernel   gather + (+1e-8) + normalise -> A, B [M, D] (+ transposed copies), row norms, the positive dot products
//   ssl_pass_kernel<0>   row sums of exp(logits) (block = 64 rows x all columns, fixed order, no atomics)
//   ssl_finish_kernel    per-row loss terms -> mean (single block, fixed order), per-row backward coefficients
//   ssl_pass_kernel<1/2> backward, logits recomputed tile by tile (flash-style): dA_j = c_j/(M T) (sum_k w_jk b_k - b_j),
//                        dB_k = 1/(M T) (sum_j c_j w_jk a_j - c_k a_k), w_jk = exp(l_jk) / deno_j; then the
//                        normalisation backward and the scatter to the table rows (atomic adds: a repeated id gets the
//                        sum of its gradients).
#include <math_constants.h>

#include "hgr_internal.cuh"

namespace hgr {

constexpr int SSL_T = 64;         // tile: 64 rows x 64 columns of logits per block step
constexpr int SSL_THREADS = 256;  // 16 x 16 threads, 4 x 4 logits each

// One warp per picked row.
__global__ void __launch_bounds__(256) ssl_prepare_kernel(const float *__restrict__ E1, const float *__restrict__ E2,
                                                          const int64_t *__restrict__ nodes, int64_t M, int64_t n_rows1,
                                                          int64_t n_rows2, int D, float add_eps, int normalize,
                                                          float *__restrict__ A, float *__restrict__ B, float *__restrict__ nrm,
                                                          float *__restrict__ pos, int32_t *__restrict__ bad, float *__restrict__ At,
                                                          float *__restrict__ Bt, int64_t Mp, float *__restrict__ act) {
    const int lane = threadIdx.x & 31;
    const int64_t j = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (j >= Mp) return;
    if (j >= M) {  // zero padding of the transposed copies up to the tile size
        for (int d = lane; d < D; d += 32) At[d * Mp + j] = Bt[d * Mp + j] = 0.f;
        if (lane == 0) act[j] = 0.f;
        return;
    }
    const int64_t r = nodes ? nodes[j] : j;
    // a NEGATIVE index marks an inactive slot (a repeated id of a fixed-size batch, loss_torch.contrastLoss_padded): it takes
    // no part in the loss; an index beyond the tables is an error and is counted
    const bool ok = r >= 0 && r < n_rows1 && r < n_rows2;
    if (!ok && r >= 0 && lane == 0) atomicAdd(bad, 1);
    if (lane == 0) act[j] = ok ? 1.f : 0.f;
    float xa[4], xb[4], sa = 0.f, sb = 0.f;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int d = lane + 32 * q;
        xa[q] = (ok && d < D) ? E1[r * D + d] + add_eps : 0.f;
        xb[q] = (ok && d < D) ? E2[r * D + d] + add_eps : 0.f;
        sa += xa[q] * xa[q];
        sb += xb[q] * xb[q];
    }
    sa = group_sum<32>(sa, 0xffffffffu);
    sb = group_sum<32>(sb, 0xffffffffu);
    const float na = normalize ? fmaxf(sqrtf(sa), 1e-12f) : 1.f, nb = normalize ? fmaxf(sqrtf(sb), 1e-12f) : 1.f;
    float dot = 0.f;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int d = lane + 32 * q;
        const float ya = xa[q] / na, yb = xb[q] / nb;
        if (d < D) {
            A[j * D + d] = ya;
            B[j * D + d] = yb;
            At[d * Mp + j] = ya;  // [D][Mp] copies: the pass kernels read 4 consecutive rows of one feature as one float4
            Bt[d * Mp + j] = yb;
        }
        dot += ya * yb;
    }
    dot = group_sum<32>(dot, 0xffffffffu);
    if (lane == 0) {
        nrm[2 * j] = na;
        nrm[2 * j + 1] = nb;
        pos[j] = dot;
    }
}

// MODE 0: rowsum[j] = sum_k exp(a_j.b_k / T)                     block owns 64 rows j, loops over column tiles
// MODE 1: GA[j, :]  = sum_k c_j exp(a_j.b_k / T) / deno_j * b_k   same ownership
// MODE 2: GB[k, :]  = sum_j c_j exp(a_j.b_k / T) / deno_j * a_j   block owns 64 columns k, loops over row tiles
// X = the owner side's table, Y = the looped side's table (MODE 2: X = B, Y = A).  Xt_g / Yt_g are their transposes
// [D][Mp] (written by ssl_prepare_kernel, Mp = M rounded up to the tile, zero padded): a thread owns 4 consecutive owner
// rows x 4 consecutive looped rows of the 64 x 64 logit tile and reads each operand as ONE 128-bit shared-memory load per
// feature (2 LDS.128 per 16 FMA; the first version read 8 scalars per 16 FMA and ran at 10 % of the fp32 rate).
template <int MODE, int D>
__global__ void __launch_bounds__(SSL_THREADS) ssl_pass_kernel(const float *__restrict__ Xt_g, const float *__restrict__ Yt_g,
                                                               const float *__restrict__ Y_g, int64_t M, int64_t Mp, float inv_temp,
                                                               const float *__restrict__ deno, const float *__restrict__ coef,
                                                               const float *__restrict__ act, float *__restrict__ out) {
    // gridDim.y blocks share an owner tile: block y takes every gridDim.y-th looped tile and writes its own partial
    // result (slice y of `out`); the consumers add the slices in order, so the sums stay deterministic.
    out += (size_t)blockIdx.y * (size_t)M * (MODE == 0 ? 1 : D);
    extern __shared__ __align__(16) float ssl_sm[];
    constexpr int DW = D / 16;    // output features per thread in the second product
    constexpr int GLD = SSL_T + 4;
    float *Xt = ssl_sm;           // [D][64] owner rows, transposed
    float *Yt = Xt + D * SSL_T;   // [D][64] looped rows, transposed
    float *Yr = Yt + D * SSL_T;   // [64][D] looped rows (MODE 1, 2)
    float *Gs = Yr + SSL_T * D;   // [64][68] weights     (MODE 1, 2)
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int64_t o0 = (int64_t)blockIdx.x * SSL_T;
    for (int e = threadIdx.x; e < D * (SSL_T / 4); e += SSL_THREADS) {
        const int d = e / (SSL_T / 4), c = e % (SSL_T / 4);
        *reinterpret_cast<float4 *>(Xt + d * SSL_T + 4 * c) = __ldg(reinterpret_cast<const float4 *>(Xt_g + d * Mp + o0) + c);
    }
    float rowsum[4] = {0.f, 0.f, 0.f, 0.f};
    float acc2[4][DW];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int m = 0; m < DW; ++m) acc2[i][m] = 0.f;
    float oscale[4] = {0.f, 0.f, 0.f, 0.f};  // MODE 1: c_j / deno_j of the owner rows
    if (MODE == 1) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int64_t j = o0 + ty * 4 + i;
            oscale[i] = j < M ? coef[j] / deno[j] : 0.f;
        }
    }
    for (int64_t l0 = (int64_t)blockIdx.y * SSL_T; l0 < M; l0 += (int64_t)gridDim.y * SSL_T) {
        __syncthreads();
        for (int e = threadIdx.x; e < D * (SSL_T / 4); e += SSL_THREADS) {
            const int d = e / (SSL_T / 4), c = e % (SSL_T / 4);
            *reinterpret_cast<float4 *>(Yt + d * SSL_T + 4 * c) = __ldg(reinterpret_cast<const float4 *>(Yt_g + d * Mp + l0) + c);
        }
        if (MODE != 0) {
            for (int e = threadIdx.x; e < SSL_T * (D / 4); e += SSL_THREADS) {
                const int r = e / (D / 4), c = e % (D / 4);
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (l0 + r < M) v = __ldg(reinterpret_cast<const float4 *>(Y_g + (l0 + r) * D) + c);
                *reinterpret_cast<float4 *>(Yr + r * D + 4 * c) = v;
            }
        }
        __syncthreads();
        // logits of owner rows {4 ty + i} against looped rows {4 tx + jj}
        float acc[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) acc[i][jj] = 0.f;
#pragma unroll 8
        for (int d = 0; d < D; ++d) {
            const float4 xa = *reinterpret_cast<const float4 *>(Xt + d * SSL_T + 4 * ty);
            const float4 yb = *reinterpret_cast<const float4 *>(Yt + d * SSL_T + 4 * tx);
            const float xv[4] = {xa.x, xa.y, xa.z, xa.w}, yv[4] = {yb.x, yb.y, yb.z, yb.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) acc[i][jj] = fmaf(xv[i], yv[jj], acc[i][jj]);
        }
        // looped rows that exist and are active (MODE 0, 1: 1 / 0); MODE 2: c_l / deno_l of the looped rows (0 when inactive)
        float lscale[4];
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
            const int64_t l = l0 + 4 * tx + jj;
            lscale[jj] = l < M ? (MODE == 2 ? coef[l] / deno[l] : act[l]) : 0.f;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            float g[4];
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) {
                const float w = lscale[jj] != 0.f ? expf(acc[i][jj] * inv_temp) : 0.f;
                if (MODE == 0) rowsum[i] += w;
                g[jj] = MODE == 1 ? w * oscale[i] : w * lscale[jj];
            }
            if (MODE != 0) *reinterpret_cast<float4 *>(Gs + (4 * ty + i) * GLD + 4 * tx) = make_float4(g[0], g[1], g[2], g[3]);
        }
        if (MODE != 0) {
            __syncthreads();
            // acc2[owner row][feature] += sum_c G[owner row][c] * Y[c][feature]
#pragma unroll 2
            for (int c0 = 0; c0 < SSL_T; c0 += 4) {
                float gv[4][4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float4 t = *reinterpret_cast<const float4 *>(Gs + (4 * ty + i) * GLD + c0);
                    gv[i][0] = t.x; gv[i][1] = t.y; gv[i][2] = t.z; gv[i][3] = t.w;
                }
#pragma unroll
                for (int cc = 0; cc < 4; ++cc) {
                    float yv[DW];
#pragma unroll
                    for (int m = 0; m < DW; ++m) yv[m] = Yr[(c0 + cc) * D + tx * DW + m];
#pragma unroll
                    for (int i = 0; i < 4; ++i)
#pragma unroll
                        for (int m = 0; m < DW; ++m) acc2[i][m] = fmaf(gv[i][cc], yv[m], acc2[i][m]);
                }
            }
        }
    }
    if (MODE == 0) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float s = group_sum<16>(rowsum[i], 0xffffffffu);  // the 16 tx lanes of a half warp share the row
            const int64_t j = o0 + 4 * ty + i;
            if (tx == 0 && j < M) out[j] = s;
        }
    } else {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int64_t j = o0 + 4 * ty + i;
            if (j < M)
#pragma unroll
                for (int m = 0; m < DW; ++m) out[j * D + tx * DW + m] = acc2[i][m];
        }
    }
}

// kind 0 (contrastLoss): deno = rowsum + 1e-8, term = log(deno) - pos / T, c = 1
// kind 1 (InfoNCE):      r = exp(pos / T) / rowsum, term = -log(r + 10e-6), c = r / (r + 10e-6)
__global__ void __launch_bounds__(1024) ssl_finish_kernel(const float *__restrict__ rowsum, int n_split, const float *__restrict__ pos,
                                                          int64_t M, float inv_temp, int kind, float *__restrict__ deno,
                                                          float *__restrict__ coef, float *__restrict__ loss,
                                                          const float *__restrict__ act, float *__restrict__ n_active) {
    __shared__ double sh[1024];
    __shared__ int cnt[1024];
    double t = 0.0;
    int na = 0;
    for (int64_t j = threadIdx.x; j < M; j += 1024) {
        if (act[j] == 0.f) {  // inactive slot: no loss term, no gradient
            deno[j] = 1.f;
            coef[j] = 0.f;
            continue;
        }
        ++na;
        float rs = rowsum[j];
        for (int s = 1; s < n_split; ++s) rs += rowsum[(int64_t)s * M + j];
        const float p = pos[j] * inv_temp;
        if (kind == 0) {
            const float dn = rs + 1e-8f;
            deno[j] = dn;
            coef[j] = 1.f;
            t += (double)(logf(dn) - p);
        } else {
            const float r = expf(p) / rs;
            deno[j] = rs;
            coef[j] = r / (r + 10e-6f);
            t += (double)(-logf(r + 10e-6f));
        }
    }
    sh[threadIdx.x] = t;
    cnt[threadIdx.x] = na;
    __syncthreads();
    for (int s = 512; s > 0; s >>= 1) {
        if ((int)threadIdx.x < s) {
            sh[threadIdx.x] += sh[threadIdx.x + s];
            cnt[threadIdx.x] += cnt[threadIdx.x + s];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        loss[0] = cnt[0] > 0 ? (float)(sh[0] / (double)cnt[0]) : 0.f;  // the mean runs over the active rows
        n_active[0] = (float)cnt[0];
    }
}

// dY_j = scale * (G_j - c_j * other_j)  with scale = grad / (M T); then the normalisation backward
// dx = (dY - y (dY . y)) / ||x|| and the store to the table row (or row j when there is no index).
__global__ void __launch_bounds__(256) ssl_scatter_kernel(const float *__restrict__ G, int n_split, const float *__restrict__ self_n,
                                                          const float *__restrict__ other_n, const float *__restrict__ coef,
                                                          const float *__restrict__ nrm, int which, const int64_t *__restrict__ nodes,
                                                          int64_t M, int64_t n_rows, int D, float inv_temp, int normalize,
                                                          const float *__restrict__ grad_out, float *__restrict__ dE,
                                                          const float *__restrict__ n_active) {
    const int lane = threadIdx.x & 31;
    const int64_t j = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (j >= M) return;
    const int64_t r = nodes ? nodes[j] : j;
    if (r < 0 || r >= n_rows) return;
    const float scale = grad_out[0] * inv_temp / fmaxf(n_active[0], 1.f);
    const float c = coef[j];
    float g[4], y[4], gy = 0.f;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int d = lane + 32 * q;
        y[q] = d < D ? self_n[j * D + d] : 0.f;
        float gs = 0.f;
        if (d < D) {
            gs = G[j * D + d];
            for (int s = 1; s < n_split; ++s) gs += G[((int64_t)s * M + j) * D + d];
        }
        g[q] = d < D ? scale * (gs - c * other_n[j * D + d]) : 0.f;
        gy += g[q] * y[q];
    }
    gy = group_sum<32>(gy, 0xffffffffu);
    const float n = nrm[2 * j + which];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int d = lane + 32 * q;
        // dE is zero-filled by the caller; with unique ids (every reference caller passes torch.unique) one add per element is
        // a store, and a caller that repeats an id gets the SUM of its gradients, like index_select's backward, instead of the last one
        if (d < D) atomicAdd(dE + r * D + d, normalize ? (g[q] - y[q] * gy) / n : g[q]);
    }
}

constexpr int SSL_MAX_SPLIT = 8;

// slices of the looped dimension: enough blocks for two waves of 148 SMs
static int ssl_splits(int64_t M) {
    const int64_t owners = ceil_div(M > 0 ? M : 1, SSL_T);
    int64_t s = ceil_div(296, owners);
    if (s > SSL_MAX_SPLIT) s = SSL_MAX_SPLIT;
    if (s > owners) s = owners;  // never more slices than looped tiles
    return (int)(s < 1 ? 1 : s);
}

struct SslWs {
    float *A, *B, *nrm, *pos, *rowsum, *deno, *coef, *G, *At, *Bt, *act, *n_active;
    int64_t Mp;  // M rounded up to the 64-row tile: leading dimension of the transposed copies
    size_t total;
};

static SslWs ssl_layout(void *base, int64_t M, int D) {
    SslWs w;
    const size_t S = (size_t)ssl_splits(M);
    size_t o = 0;
    auto take = [&](size_t n) {
        float *p = base ? reinterpret_cast<float *>(static_cast<uint8_t *>(base) + o) : nullptr;
        o += (n * sizeof(float) + 255) / 256 * 256;
        return p;
    };
    const size_t m = (size_t)(M > 0 ? M : 1);
    w.A = take(m * D);
    w.B = take(m * D);
    w.nrm = take(2 * m);
    w.pos = take(m);
    w.rowsum = take(m * S);
    w.deno = take(m);
    w.coef = take(m);
    w.G = take(m * D * S);
    w.Mp = (int64_t)ceil_div((int64_t)m, SSL_T) * SSL_T;
    w.At = take((size_t)w.Mp * D);
    w.Bt = take((size_t)w.Mp * D);
    w.act = take((size_t)w.Mp);
    w.n_active = take(1);
    w.total = o;
    return w;
}

template <int MODE>
static int launch_pass(int D, const float *Xt, const float *Yt, const float *Y, int64_t M, int64_t Mp, float inv_temp, const float *deno,
                       const float *coef, const float *act, float *out, cudaStream_t st) {
    const dim3 grid((unsigned)ceil_div(M, SSL_T), (unsigned)ssl_splits(M));
    if (grid.x == 0) return HGR_OK;
#define HGR_SSL_LAUNCH(DD)                                                                                                 \
    {                                                                                                                      \
        const size_t smem = (size_t)(MODE == 0 ? 2 * SSL_T * DD : 3 * SSL_T * DD + SSL_T * (SSL_T + 4)) * sizeof(float);     \
        HGR_CUDA_OK(cudaFuncSetAttribute(ssl_pass_kernel<MODE, DD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        ssl_pass_kernel<MODE, DD><<<grid, SSL_THREADS, smem, st>>>(Xt, Yt, Y, M, Mp, inv_temp, deno, coef, act, out);      \
    }
    if (D == 32) HGR_SSL_LAUNCH(32)
    else if (D == 64) HGR_SSL_LAUNCH(64)
    else HGR_SSL_LAUNCH(128)
#undef HGR_SSL_LAUNCH
    HGR_LAUNCH_OK("ssl_pass_kernel");
    return HGR_OK;
}

}  // namespace hgr

extern "C" {

size_t hgr_ssl_workspace_bytes(int64_t M, int32_t D) { return hgr::ssl_layout(nullptr, M, D).total; }

int hgr_ssl_loss_fwd_f32(const float *E1, const float *E2, int64_t n_rows1, int64_t n_rows2, int32_t D, const int64_t *nodes,
                         int64_t M, float temp, int32_t kind, int32_t normalize, float *loss, void *saved, size_t saved_bytes,
                         int32_t *bad_index_count, hgr_stream_t stream) {
    using namespace hgr;
    cudaStream_t st = (cudaStream_t)stream;
    HGR_REQUIRE(D == 32 || D == 64 || D == 128, "D = %d unsupported (32, 64 or 128)", D);
    HGR_REQUIRE(kind == 0 || kind == 1, "kind %d unknown (0 contrastLoss, 1 InfoNCE)", kind);
    HGR_REQUIRE(temp > 0.f, "temperature must be positive");
    HGR_REQUIRE(M >= 0 && E1 && E2 && loss && bad_index_count, "NULL argument or negative M");
    const SslWs w = ssl_layout(saved, M, D);
    if (saved == nullptr || saved_bytes < w.total)
        return set_error(HGR_ERR_WORKSPACE, "ssl workspace: need %zu bytes, got %zu", w.total, saved_bytes);
    HGR_REQUIRE((reinterpret_cast<uintptr_t>(saved) & 255u) == 0, "workspace must be 256-byte aligned");
    const float inv_temp = 1.0f / temp;
    if (M > 0) {
        ssl_prepare_kernel<<<(unsigned)ceil_div(w.Mp, 8), 256, 0, st>>>(E1, E2, nodes, M, n_rows1, n_rows2, D, kind == 0 ? 1e-8f : 0.f,
                                                                       normalize, w.A, w.B, w.nrm, w.pos, bad_index_count, w.At, w.Bt, w.Mp, w.act);
        HGR_LAUNCH_OK("ssl_prepare_kernel");
        int rc = launch_pass<0>(D, w.At, w.Bt, w.B, M, w.Mp, inv_temp, nullptr, nullptr, w.act, w.rowsum, st);
        if (rc) return rc;
    }
    ssl_finish_kernel<<<1, 1024, 0, st>>>(w.rowsum, ssl_splits(M), w.pos, M, inv_temp, kind, w.deno, w.coef, loss, w.act, w.n_active);
    HGR_LAUNCH_OK("ssl_finish_kernel");
    return HGR_OK;
}

int hgr_ssl_loss_bwd_f32(int64_t n_rows1, int64_t n_rows2, int32_t D, const int64_t *nodes, int64_t M, float temp, int32_t normalize,
                         void *saved, size_t saved_bytes, const float *grad_out, float *dE1, float *dE2, hgr_stream_t stream) {
    using namespace hgr;
    cudaStream_t st = (cudaStream_t)stream;
    HGR_REQUIRE(D == 32 || D == 64 || D == 128, "D = %d unsupported (32, 64 or 128)", D);
    HGR_REQUIRE(M >= 0 && grad_out && saved, "NULL argument or negative M");
    const SslWs w = ssl_layout(saved, M, D);
    HGR_REQUIRE(saved_bytes >= w.total, "ssl workspace too small");
    if (M == 0) return HGR_OK;
    const float inv_temp = 1.0f / temp;
    if (dE1) {
        int rc = launch_pass<1>(D, w.At, w.Bt, w.B, M, w.Mp, inv_temp, w.deno, w.coef, w.act, w.G, st);
        if (rc) return rc;
        ssl_scatter_kernel<<<(unsigned)ceil_div(M, 8), 256, 0, st>>>(w.G, ssl_splits(M), w.A, w.B, w.coef, w.nrm, 0, nodes, M, n_rows1, D, inv_temp,
                                                                    normalize, grad_out, dE1, w.n_active);
        HGR_LAUNCH_OK("ssl_scatter_kernel");
    }
    if (dE2) {
        int rc = launch_pass<2>(D, w.Bt, w.At, w.A, M, w.Mp, inv_temp, w.deno, w.coef, w.act, w.G, st);
        if (rc) return rc;
        ssl_scatter_kernel<<<(unsigned)ceil_div(M, 8), 256, 0, st>>>(w.G, ssl_splits(M), w.B, w.A, w.coef, w.nrm, 1, nodes, M, n_rows2, D, inv_temp,
                                                                    normalize, grad_out, dE2, w.n_active);
        HGR_LAUNCH_OK("ssl_scatter_kernel");
    }
    return HGR_OK;
}

}  // extern "C"
