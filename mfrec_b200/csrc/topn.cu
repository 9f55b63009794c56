// Top-N scoring: rows of U.V^T (+ the predictor's affine / logistic map), masked, ranked.
//
// Replaces the per-item Python loops of MFRecommender.find_recommended_items
// (mfrec/recommendation/mf.py:144-193) and GDRecommender.find_user_top_match
// (gradient_descent.py:769-802) for a batch of users.  Semantics kept, quirks included:
//   * candidates are item ids [0, n_candidates)  (mf.py scores the enumeration index);
//   * the user's rated items AND the item whose id equals the user id are excluded
//     (mf.py:161-162, gradient_descent.py:778-779 append user_index to the rated list);
//   * NaN scores become 0, exact zeros are dropped (mf.py:176-181);
//   * order: score descending, ties by ascending item id (Python's stable sort), first N.
//
// This file is the EXACT path: fp32 scores from a shared-memory tiled SGEMM on the CUDA cores,
// one 64-bit key per (user, item) = (order-preserving score bits, ~item), a segmented radix sort
// per user and a gather of the first N.  It is what the parity tests pin; the tensor-core
// (tcgen05) scoring stage for the all-users x all-items sweep builds on the same key / mask /
// selection stages (DESIGN.md).
#include <cub/device/device_segmented_radix_sort.cuh>

#include "common.cuh"

namespace {

struct TopnParams {
    const float *P, *Q, *ib, *ub;
    const int32_t *users;   // [nub] user ids of this batch
    int nub, nc, kpad;
    int predictor;
    float mu, min_rating, max_rating;
    uint64_t *keys;         // [nub][nc]
};

// C[64 users][64 items] per CTA, 256 threads, 4x4 outputs per thread, K tiles of 16
__global__ void __launch_bounds__(256) topn_score_kernel(const TopnParams p)
{
    __shared__ float As[16][64 + 4];
    __shared__ float Bs[16][64 + 4];
    __shared__ int32_t urow[64];
    const int tid = threadIdx.x;
    const int u0 = blockIdx.y * 64, i0 = blockIdx.x * 64;
    if (tid < 64) urow[tid] = (u0 + tid < p.nub) ? p.users[u0 + tid] : -1;
    __syncthreads();
    const int tx = tid & 15, ty = tid >> 4;       // 16 x 16 threads
    float acc[4][4] = {};
    const int lr = tid >> 2, lc = (tid & 3) * 4;  // loader: row 0..63, k offset 0,4,8,12
    for (int k0 = 0; k0 < p.kpad; k0 += 16) {
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
        const int ur = urow[lr];
        if (ur >= 0) a = *reinterpret_cast<const float4 *>(p.P + (size_t)ur * p.kpad + k0 + lc);
        if (i0 + lr < p.nc) b = *reinterpret_cast<const float4 *>(p.Q + (size_t)(i0 + lr) * p.kpad + k0 + lc);
        As[lc + 0][lr] = a.x; As[lc + 1][lr] = a.y; As[lc + 2][lr] = a.z; As[lc + 3][lr] = a.w;
        Bs[lc + 0][lr] = b.x; Bs[lc + 1][lr] = b.y; Bs[lc + 2][lr] = b.z; Bs[lc + 3][lr] = b.w;
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < 16; ++kk) {
            float av[4], bv[4];
#pragma unroll
            for (int r = 0; r < 4; ++r) { av[r] = As[kk][ty * 4 + r]; bv[r] = Bs[kk][tx * 4 + r]; }
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[r][c] = fmaf(av[r], bv[c], acc[r][c]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int ul = u0 + ty * 4 + r;
        if (ul >= p.nub) continue;
        const int ur = urow[ty * 4 + r];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int it = i0 + tx * 4 + c;
            if (it >= p.nc) continue;
            const float dot = acc[r][c];
            const float bsum = p.ib[it] + p.ub[ur];
            float s;
            switch (p.predictor) {
            case MFREC_PRED_GD_RATING: s = dot + 1.0f; break;
            case MFREC_PRED_GD_RATING_BIAS: s = dot + (p.mu + bsum); break;
            case MFREC_PRED_KMF_LINEAR: s = dot + bsum; break;
            case MFREC_PRED_KMF_LOGISTIC:
                s = p.min_rating + (1.f / (1.f + expf(-(dot + bsum)))) * (p.max_rating - p.min_rating);
                break;
            case MFREC_PRED_KMF_LINEAR_NEG: s = p.min_rating + (dot + bsum) * (p.max_rating - p.min_rating); break;
            default: s = dot; break;
            }
            uint64_t key = 0;   // 0 = excluded (sorts last)
            if (s == s && s != 0.f && it != ur)   // NaN -> 0 -> dropped; zeros dropped; id quirk
                key = ((uint64_t)order_bits(s) << 32) | (uint32_t)(~(uint32_t)it);
            p.keys[(size_t)ul * p.nc + it] = key;
        }
    }
}

__global__ void topn_mask_kernel(const int64_t *__restrict__ indptr, const int32_t *__restrict__ rated,
                                 int u_first, int nub, int nc, uint64_t *__restrict__ keys)
{
    // one warp per user row
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= nub) return;
    const int64_t a = indptr[u_first + row], b = indptr[u_first + row + 1];
    for (int64_t j = a + (threadIdx.x & 31); j < b; j += 32) {
        const int it = rated[j];
        if (it >= 0 && it < nc) keys[(size_t)row * nc + it] = 0;
    }
}

__global__ void topn_gather_kernel(const uint64_t *__restrict__ sorted, int nub, int nc, int N,
                                   int32_t *__restrict__ items, double *__restrict__ scores,
                                   int32_t *__restrict__ counts)
{
    const int row = blockIdx.x;
    int cnt = 0;
    for (int j = threadIdx.x; j < N; j += blockDim.x) {
        const uint64_t key = j < nc ? sorted[(size_t)row * nc + j] : 0;
        if (key) {
            items[(size_t)row * N + j] = (int32_t)(~(uint32_t)(key & 0xffffffffu));
            scores[(size_t)row * N + j] = (double)unorder_bits((uint32_t)(key >> 32));
        } else {
            items[(size_t)row * N + j] = -1;
            scores[(size_t)row * N + j] = 0.0;
        }
        cnt += key != 0;
    }
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    __shared__ int tot;
    if (threadIdx.x == 0) tot = 0;
    __syncthreads();
    if ((threadIdx.x & 31) == 0) atomicAdd(&tot, cnt);
    __syncthreads();
    if (threadIdx.x == 0) counts[row] = tot;
}

__global__ void iota_offsets_kernel(int64_t *off, int n, int64_t stride)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i <= n) off[i] = (int64_t)i * stride;
}

}  // namespace

extern "C" int mfrec_topn(mfrec_ctx *ctx, int predictor, int k, const double *u, const double *v,
                          int32_t ni, int32_t nu, const int32_t *users, int32_t n_users,
                          int32_t n_candidates, const int64_t *rated_indptr, const int32_t *rated_items,
                          double mu, const double *items_bias, const double *users_bias,
                          double min_rating, double max_rating, int32_t N, int32_t *out_items,
                          double *out_scores, int32_t *out_counts)
{
    if (!ctx || !u || !v) return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_topn: NULL argument");
    if (n_users <= 0 || n_candidates <= 0 || N <= 0)   // nothing to score: no upload either
        return mfrec_topn_on_model(ctx, nullptr, predictor, users, n_users, n_candidates, rated_indptr, rated_items, mu,
                                min_rating, max_rating, N, out_items, out_scores, out_counts, ni, nu);
    mfrec_model *M = nullptr;
    MF_TRY(mfrec_model_create(ctx, nullptr, k, ni, nu, u, v, items_bias, users_bias, &M));
    const int rc = mfrec_topn_on_model(ctx, M, predictor, users, n_users, n_candidates, rated_indptr, rated_items, mu,
                                    min_rating, max_rating, N, out_items, out_scores, out_counts, ni, nu);
    mfrec_model_destroy(M);
    return rc;
}

// ni / nu: only read when M is NULL (argument checks of a call that scores nothing)
int mfrec_topn_on_model(mfrec_ctx *ctx, const mfrec_model *M, int predictor, const int32_t *users, int32_t n_users,
                     int32_t n_candidates, const int64_t *rated_indptr, const int32_t *rated_items, double mu,
                     double min_rating, double max_rating, int32_t N, int32_t *out_items, double *out_scores,
                     int32_t *out_counts, int32_t ni, int32_t nu)
{
    if (M) { ni = M->ni; nu = M->nu; }
    if (!ctx || !users || !out_items || !out_scores || !out_counts)
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_topn: NULL argument");
    if (M && (M->user_perm || M->item_perm))
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_topn: the model must be in identity layout (created without a ratings layout)");
    if (predictor < 0 || predictor > MFREC_PRED_DOT || n_users < 0 || N <= 0 || n_candidates < 0 ||
        n_candidates > ni)
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_topn: predictor=%d n_users=%d N=%d n_candidates=%d",
                               predictor, n_users, N, n_candidates);
    for (int32_t j = 0; j < n_users; ++j)
        if (users[j] < 0 || users[j] >= nu)
            return mfrec_set_error(ctx, MFREC_ERR_INDEX, "mfrec_topn: user %d outside [0,%d)", users[j], nu);
    if (n_users == 0) return MFREC_OK;
    MF_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const int nc = n_candidates;
    if (nc == 0) {
        for (int64_t j = 0; j < (int64_t)n_users * N; ++j) { out_items[j] = -1; out_scores[j] = 0.0; }
        for (int32_t j = 0; j < n_users; ++j) out_counts[j] = 0;
        return MFREC_OK;
    }
    if (!M) return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_topn: NULL model");

    // batch users so the two key buffers stay under ~1 GiB each
    const int64_t max_rows = std::max<int64_t>(64, (int64_t)(1ll << 27) / nc);
    const int batch = (int)std::min<int64_t>(n_users, max_rows);
    DevBuf<uint64_t> keys_a, keys_b;
    DevBuf<int64_t> d_off, d_indptr;
    DevBuf<int32_t> d_users, d_rated, d_items, d_counts;
    DevBuf<double> d_scores;
    DevBuf<char> tmp;
    MF_CUDA(ctx, keys_a.alloc((size_t)batch * nc, ctx->stream));
    MF_CUDA(ctx, keys_b.alloc((size_t)batch * nc, ctx->stream));
    MF_CUDA(ctx, d_off.alloc((size_t)batch + 1, ctx->stream));
    MF_CUDA(ctx, d_users.alloc(n_users, ctx->stream));
    MF_CUDA(ctx, d_items.alloc((size_t)batch * N, ctx->stream));
    MF_CUDA(ctx, d_scores.alloc((size_t)batch * N, ctx->stream));
    MF_CUDA(ctx, d_counts.alloc(batch, ctx->stream));
    MF_CUDA(ctx, cudaMemcpyAsync(d_users.p, users, (size_t)n_users * 4, cudaMemcpyHostToDevice, st));
    const int64_t n_rated = rated_indptr ? rated_indptr[n_users] : 0;
    if (rated_indptr && n_rated > 0) {
        if (!rated_items) return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_topn: rated_items is NULL");
        MF_CUDA(ctx, d_indptr.alloc((size_t)n_users + 1, ctx->stream));
        MF_CUDA(ctx, d_rated.alloc((size_t)n_rated, ctx->stream));
        MF_CUDA(ctx, cudaMemcpyAsync(d_indptr.p, rated_indptr, ((size_t)n_users + 1) * 8, cudaMemcpyHostToDevice, st));
        MF_CUDA(ctx, cudaMemcpyAsync(d_rated.p, rated_items, (size_t)n_rated * 4, cudaMemcpyHostToDevice, st));
    }
    iota_offsets_kernel<<<(batch + 256) / 256, 256, 0, st>>>(d_off.p, batch, nc);
    MF_LAUNCH_CHECK(ctx);
    size_t tmp_bytes = 0;
    cub::DoubleBuffer<uint64_t> dk(keys_a.p, keys_b.p);
    MF_CUDA(ctx, cub::DeviceSegmentedRadixSort::SortKeysDescending(nullptr, tmp_bytes, dk, (int64_t)batch * nc, batch,
                                                                   d_off.p, d_off.p + 1, 0, 64, st));
    MF_CUDA(ctx, tmp.alloc(tmp_bytes, ctx->stream));

    TopnParams prm;
    prm.P = M->P; prm.Q = M->Q; prm.ib = M->ib; prm.ub = M->ub;
    prm.nc = nc; prm.kpad = M->kpad; prm.predictor = predictor;
    prm.mu = (float)mu; prm.min_rating = (float)min_rating; prm.max_rating = (float)max_rating;
    for (int first = 0; first < n_users; first += batch) {
        const int nub = std::min(batch, n_users - first);
        prm.users = d_users.p + first;
        prm.nub = nub;
        prm.keys = keys_a.p;
        dim3 grid((nc + 63) / 64, (nub + 63) / 64);
        topn_score_kernel<<<grid, 256, 0, st>>>(prm);
        MF_LAUNCH_CHECK(ctx);
        if (d_rated.p) {
            topn_mask_kernel<<<(nub + 7) / 8, 256, 0, st>>>(d_indptr.p, d_rated.p, first, nub, nc, keys_a.p);
            MF_LAUNCH_CHECK(ctx);
        }
        cub::DoubleBuffer<uint64_t> db(keys_a.p, keys_b.p);
        MF_CUDA(ctx, cub::DeviceSegmentedRadixSort::SortKeysDescending(tmp.p, tmp_bytes, db, (int64_t)nub * nc, nub,
                                                                       d_off.p, d_off.p + 1, 0, 64, st));
        ctx->launches += 8;
        topn_gather_kernel<<<nub, 128, 0, st>>>(db.Current(), nub, nc, N, d_items.p, d_scores.p, d_counts.p);
        MF_LAUNCH_CHECK(ctx);
        MF_CUDA(ctx, cudaMemcpyAsync(out_items + (size_t)first * N, d_items.p, (size_t)nub * N * 4, cudaMemcpyDeviceToHost, st));
        MF_CUDA(ctx, cudaMemcpyAsync(out_scores + (size_t)first * N, d_scores.p, (size_t)nub * N * 8, cudaMemcpyDeviceToHost, st));
        MF_CUDA(ctx, cudaMemcpyAsync(out_counts + first, d_counts.p, (size_t)nub * 4, cudaMemcpyDeviceToHost, st));
        MF_CUDA(ctx, cudaStreamSynchronize(st));
    }
    return MFREC_OK;
}

extern "C" int mfrec_model_topn(mfrec_ctx *ctx, const mfrec_model *m, int predictor, const int32_t *users,
                                int32_t n_users, int32_t n_candidates, const int64_t *rated_indptr,
                                const int32_t *rated_items, double mu, double min_rating, double max_rating,
                                int32_t N, int32_t *out_items, double *out_scores, int32_t *out_counts)
{
    if (!m) return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_model_topn: NULL model");
    return mfrec_topn_on_model(ctx, m, predictor, users, n_users, n_candidates, rated_indptr, rated_items, mu,
                               min_rating, max_rating, N, out_items, out_scores, out_counts, m->ni, m->nu);
}
