// Evaluation kernels: batched predict / RMSE over (user, item) pairs and the bias statistics
// that precede training.  All HBM-bound: one warp per pair, both factor rows read with
// coalesced 128-bit loads, shuffle-reduced dot product.
//
// Reference being replaced (all interpreted Python loops, one k-dot per call):
//   metrics.test_predict_rating            mfrec/recommendation/metrics.py:51-82
//   GDRecommender.predict_rating[_with_bias]  gradient_descent.py:621-648
//   KMFRecommender.predict_{logistic,linear,linear_neg}  kmf.py:79-103
//   compute_overall_avg base.py:504-508, compute_{items,users}_bias_bk mf.py:78-121
#include <algorithm>
#include <cmath>
#include <type_traits>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "common.cuh"

namespace {

struct PredParams {
    const float *Q, *ib, *ub;
    const void *P;   // user-factor rows: float, __half or __nv_bfloat16 (mfrec_model::p_kind)
    const int32_t *user_perm, *item_perm;
    const int32_t *pairs;
    const void *real;
    int real_is_f32;
    int64_t n;
    int predictor;
    float mu, min_rating, max_rating;
    double *out;        // nullable
    double *part;       // [gridDim.x][3]  sum e^2, sum |e|, n_valid   (nullable)
    int32_t ni, nu;
    int32_t *bad;
};

// A warp scores FOUR pairs per iteration: eight row requests (4 x 512 B at k = 128 for P and Q
// each) are in flight before the first is consumed -- with one pair at a time the kernel waited
// out two dependent L2 round trips per pair (ncu r02m: 3.9 G pairs/s, 1.2 TB/s of DRAM) -- and
// lanes 0..3 finish one pair each (bias lookup, predictor map, error) instead of lane 0 doing all.
// PT: storage type of the user-factor rows (float; __half / __nv_bfloat16 for a model trained with
// mfrec_opts.storage): 16-bit rows are widened in registers, the arithmetic is float32.
template <int V, typename PT>
__device__ __forceinline__ void load_p(float (&x)[V], const void *P, int64_t elem)
{
    const PT *p = static_cast<const PT *>(P) + elem;
    if constexpr (sizeof(PT) == 4) {
        if constexpr (V == 4) { const float4 t = *reinterpret_cast<const float4 *>(p); x[0] = t.x; x[1] = t.y; x[2] = t.z; x[3] = t.w; }
        else if constexpr (V == 2) { const float2 t = *reinterpret_cast<const float2 *>(p); x[0] = t.x; x[1] = t.y; }
        else x[0] = *reinterpret_cast<const float *>(p);
    } else {
        uint32_t w[(V + 1) / 2];
        if constexpr (V == 4) { const uint2 t = *reinterpret_cast<const uint2 *>(p); w[0] = t.x; w[1] = t.y; }
        else if constexpr (V == 2) w[0] = *reinterpret_cast<const uint32_t *>(p);
        else w[0] = *reinterpret_cast<const uint16_t *>(p);
#pragma unroll
        for (int h = 0; h < V; ++h) {
            const uint32_t bits = (h & 1) ? (w[h / 2] >> 16) : (w[h / 2] & 0xffffu);
            if constexpr (std::is_same<PT, __half>::value) x[h] = __half2float(__ushort_as_half((unsigned short)bits));
            else x[h] = __uint_as_float(bits << 16);
        }
    }
}

// (4 CTAs of 256 threads per SM = 64 registers: measured best -- 3 CTAs at 78 registers 9.5 ms per 50 M pairs,
// 4 at 64 6.9 ms, 5 at 48 with spills 7.8 ms)
template <int E, typename PT>
__global__ void __launch_bounds__(256, 4) predict_kernel(const PredParams p)
{
    constexpr int KPAD = E * 32;
    constexpr int V = E >= 4 ? 4 : E, NV = E / V;
    constexpr int G4 = 4;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
    double s2 = 0.0, s1 = 0.0, cnt = 0.0;
    // Three dependent round trips per group of pairs -- pair ids, their packed row numbers, the rows --
    // made the kernel wait out three latencies per iteration (ncu r02w: 65 % long-scoreboard stalls,
    // 6 TB/s).  The ids of the NEXT group are requested before this group's rows and turned into row
    // numbers after this group's dot products, so an iteration waits for one latency, the rows'.
    int2 ui_n[G4];
    bool ok_n[G4];
    auto request_pairs = [&](int64_t j0) {
#pragma unroll
        for (int t = 0; t < G4; ++t) {
            const int64_t j = j0 + t;
            ui_n[t] = make_int2(0, 0);
            ok_n[t] = j < p.n;
            if (ok_n[t]) ui_n[t] = reinterpret_cast<const int2 *>(p.pairs)[j];
        }
    };
    int32_t ur_n[G4], ir_n[G4];   // (packed row numbers: < 2^27)
    auto resolve_rows = [&]() {
#pragma unroll
        for (int t = 0; t < G4; ++t) {
            const int2 ui = ui_n[t];
            if (ok_n[t] && (ui.x < 0 || ui.x >= p.nu || ui.y < 0 || ui.y >= p.ni)) {
                if (lane == 0) atomicOr(p.bad, 1);
                ok_n[t] = false;
            }
            ur_n[t] = ok_n[t] ? (p.user_perm ? p.user_perm[ui.x] : ui.x) : 0;
            ir_n[t] = ok_n[t] ? (p.item_perm ? p.item_perm[ui.y] : ui.y) : 0;
        }
    };
    const int64_t j_first = ((int64_t)blockIdx.x * (blockDim.x >> 5) + wib) * G4;
    request_pairs(j_first);
    resolve_rows();
    for (int64_t j0 = j_first; j0 < p.n; j0 += warps * G4) {
        int32_t ur[G4], ir[G4];
        bool ok[G4];
#pragma unroll
        for (int t = 0; t < G4; ++t) { ur[t] = ur_n[t]; ir[t] = ir_n[t]; ok[t] = ok_n[t]; }
        request_pairs(j0 + warps * G4);   // (past the end: nothing is loaded, every ok_n is false)
        float part[G4];
#pragma unroll
        for (int t = 0; t < G4; ++t) part[t] = 0.f;
#pragma unroll
        for (int c = 0; c < NV; ++c) {
            const int off = (c * 32 + lane) * V;
            float a[G4][V], b[G4][V];
#pragma unroll
            for (int t = 0; t < G4; ++t) {
                load_p<V, PT>(a[t], p.P, (int64_t)ur[t] * KPAD + off);
                load_p<V, float>(b[t], p.Q, (int64_t)ir[t] * KPAD + off);
            }
#pragma unroll
            for (int t = 0; t < G4; ++t)
#pragma unroll
                for (int h = 0; h < V; ++h) part[t] = fmaf(a[t][h], b[t][h], part[t]);
        }
        resolve_rows();   // the next group's row numbers: their loads overlap the reduction and the finish below
#pragma unroll
        for (int o = 16; o > 0; o >>= 1)
#pragma unroll
            for (int t = 0; t < G4; ++t) part[t] += __shfl_xor_sync(0xffffffffu, part[t], o);
        if (lane < G4) {
            // lane t finishes pair t (every lane holds all four sums after the butterfly)
            const float dot = lane == 0 ? part[0] : lane == 1 ? part[1] : lane == 2 ? part[2] : part[3];
            const bool mine_ok = lane == 0 ? ok[0] : lane == 1 ? ok[1] : lane == 2 ? ok[2] : ok[3];
            const int64_t u_ = lane == 0 ? ur[0] : lane == 1 ? ur[1] : lane == 2 ? ur[2] : ur[3];
            const int64_t i_ = lane == 0 ? ir[0] : lane == 1 ? ir[1] : lane == 2 ? ir[2] : ir[3];
            const int64_t j = j0 + lane;
            if (mine_ok) {
                const float bsum = p.ib[i_] + p.ub[u_];
                float pred;
                switch (p.predictor) {
                case MFREC_PRED_GD_RATING: pred = dot + 1.0f; break;
                case MFREC_PRED_GD_RATING_BIAS: pred = dot + (p.mu + bsum); break;
                case MFREC_PRED_KMF_LINEAR: pred = dot + bsum; break;
                case MFREC_PRED_KMF_LOGISTIC:
                    pred = p.min_rating + (1.f / (1.f + expf(-(dot + bsum)))) * (p.max_rating - p.min_rating);
                    break;
                case MFREC_PRED_KMF_LINEAR_NEG:
                    pred = p.min_rating + (dot + bsum) * (p.max_rating - p.min_rating);
                    break;
                default: pred = dot; break;
                }
                if (p.out) p.out[j] = (double)pred;
                if (p.real) {
                    const double real = p.real_is_f32 ? (double)((const float *)p.real)[j]
                                                      : ((const double *)p.real)[j];
                    const double e = real - (double)pred;
                    if (e == e) { s2 += e * e; s1 += fabs(e); cnt += 1.0; }
                }
            }
        }
    }
    if (p.part) {
        // lanes 0..3 of every warp hold partial sums: fixed-order reduction (deterministic)
        __shared__ double sh[8][4][3];
        if (lane < G4) { sh[wib][lane][0] = s2; sh[wib][lane][1] = s1; sh[wib][lane][2] = cnt; }
        __syncthreads();
        if (threadIdx.x == 0) {
            double a = 0, b = 0, c = 0;
            for (int w = 0; w < (int)(blockDim.x >> 5); ++w)
                for (int l = 0; l < G4; ++l) { a += sh[w][l][0]; b += sh[w][l][1]; c += sh[w][l][2]; }
            p.part[blockIdx.x * 3 + 0] = a;
            p.part[blockIdx.x * 3 + 1] = b;
            p.part[blockIdx.x * 3 + 2] = c;
        }
    }
}

__global__ void __launch_bounds__(256) stats_reduce_kernel(const double *__restrict__ part, int nblk,
                                                           double *__restrict__ out)
{
    __shared__ double sh[256][3];
    double a = 0, b = 0, c = 0;
    for (int i = threadIdx.x; i < nblk; i += 256) { a += part[i * 3]; b += part[i * 3 + 1]; c += part[i * 3 + 2]; }
    sh[threadIdx.x][0] = a; sh[threadIdx.x][1] = b; sh[threadIdx.x][2] = c;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o)
            for (int q = 0; q < 3; ++q) sh[threadIdx.x][q] += sh[threadIdx.x + o][q];
        __syncthreads();
    }
    if (threadIdx.x == 0) { out[0] = sh[0][0]; out[1] = sh[0][1]; out[2] = sh[0][2]; out[3] = 0.0; }
}

// ---- bias statistics ----------------------------------------------------------------------
__global__ void sum_ratings_kernel(const double *__restrict__ r, int64_t nnz, double *__restrict__ part)
{
    __shared__ double sh[256];
    double acc = 0.0;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; n < nnz; n += stride) acc += r[n];
    sh[threadIdx.x] = acc;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) part[blockIdx.x] = sh[0];
}

// Deterministic segmented sums (no floating-point atomics: the result must not depend on
// scheduling -- SURVEY T7 asks for run-to-run identical results for a fixed seed).  Ratings are
// stably sorted by segment id (item, then user), so each segment's terms sit in input order;
// one warp sums a segment with a fixed lane-strided order and a shuffle tree.
__global__ void seg_key_kernel(const int32_t *__restrict__ idx, int64_t nnz, int which, int32_t ni, int32_t nu,
                               uint32_t *__restrict__ keys, uint32_t *__restrict__ pos,
                               int32_t *__restrict__ cnt, int32_t *__restrict__ bad)
{
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; n < nnz; n += stride) {
        const int2 ui = reinterpret_cast<const int2 *>(idx)[n];
        if (ui.x < 0 || ui.x >= nu || ui.y < 0 || ui.y >= ni) {
            atomicOr(bad, 1);
            keys[n] = 0;
            pos[n] = (uint32_t)n;
            continue;
        }
        const int32_t key = which ? ui.x : ui.y;
        keys[n] = (uint32_t)key;
        pos[n] = (uint32_t)n;
        atomicAdd(&cnt[key], 1);   // integer: exact whatever the order
    }
}

__global__ void __launch_bounds__(256)
seg_bias_kernel(const uint32_t *__restrict__ pos_sorted, const int64_t *__restrict__ seg_off, int32_t n_seg,
                const int32_t *__restrict__ idx, const double *__restrict__ r, double mu,
                const double *__restrict__ bias_i,   // null: item pass (terms r - mu); else user pass (r - mu - b_i)
                double K, double *__restrict__ out)
{
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (warp >= n_seg) return;
    const int64_t a = seg_off[warp], b = seg_off[warp + 1];
    double acc = 0.0;
    for (int64_t j = a + lane; j < b; j += 32) {
        const uint32_t n = pos_sorted[j];
        double t = r[n] - mu;
        if (bias_i) t -= bias_i[idx[2 * (int64_t)n + 1]];
        acc += t;
    }
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) out[warp] = b > a ? acc / (K + (double)(b - a)) : 0.0;
}

__global__ void cnt_to_i64_kernel(const int32_t *__restrict__ cnt, int32_t n, int64_t *__restrict__ out)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i <= n) out[i] = i < n ? cnt[i] : 0;
}

// bias[seg] = sum over the segment's ratings of (r - mu [- b_i]) / (K + count), segments = items
// (which = 0) or users (which = 1)
int segmented_bias(mfrec_ctx *ctx, const int32_t *d_idx, const double *d_r, int64_t nnz, int32_t ni, int32_t nu,
                   int which, double mu, const double *bias_i, double K, double *d_out, int32_t *d_bad)
{
    cudaStream_t st = ctx->stream;
    const int32_t n_seg = which ? nu : ni;
    const int grid = ctx->sm_count * 8;
    DevBuf<uint32_t> ka, kb, va, vb;
    DevBuf<int32_t> cnt;
    DevBuf<int64_t> cnt64, off;
    MF_CUDA(ctx, ka.alloc(nnz, st)); MF_CUDA(ctx, kb.alloc(nnz, st));
    MF_CUDA(ctx, va.alloc(nnz, st)); MF_CUDA(ctx, vb.alloc(nnz, st));
    MF_CUDA(ctx, cnt.alloc((size_t)n_seg + 1, st));
    MF_CUDA(ctx, cnt64.alloc((size_t)n_seg + 1, st));
    MF_CUDA(ctx, off.alloc((size_t)n_seg + 1, st));
    MF_CUDA(ctx, cudaMemsetAsync(cnt.p, 0, ((size_t)n_seg + 1) * 4, st));
    seg_key_kernel<<<grid, 256, 0, st>>>(d_idx, nnz, which, ni, nu, ka.p, va.p, cnt.p, d_bad);
    MF_LAUNCH_CHECK(ctx);
    int bits = 1;
    while ((1ll << bits) < n_seg) ++bits;
    cub::DoubleBuffer<uint32_t> dk(ka.p, kb.p), dv(va.p, vb.p);
    size_t tmp_bytes = 0, tmp2 = 0;
    MF_CUDA(ctx, cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, dk, dv, nnz, 0, bits, st));
    MF_CUDA(ctx, cub::DeviceScan::ExclusiveSum(nullptr, tmp2, cnt64.p, off.p, n_seg + 1, st));
    DevBuf<char> tmp;
    MF_CUDA(ctx, tmp.alloc(std::max(tmp_bytes, tmp2), st));
    MF_CUDA(ctx, cub::DeviceRadixSort::SortPairs(tmp.p, tmp_bytes, dk, dv, nnz, 0, bits, st));   // stable (LSD)
    cnt_to_i64_kernel<<<(n_seg + 256) / 256, 256, 0, st>>>(cnt.p, n_seg, cnt64.p);
    MF_LAUNCH_CHECK(ctx);
    MF_CUDA(ctx, cub::DeviceScan::ExclusiveSum(tmp.p, tmp2, cnt64.p, off.p, n_seg + 1, st));
    ctx->launches += (bits + 7) / 8 * 2 + 3;
    seg_bias_kernel<<<(unsigned)ceil_div64((int64_t)n_seg * 32, 256), 256, 0, st>>>(dv.Current(), off.p, n_seg, d_idx,
                                                                                   d_r, mu, bias_i, K, d_out);
    MF_LAUNCH_CHECK(ctx);
    MF_CUDA(ctx, cudaStreamSynchronize(st));   // scratch goes back to the pool on return
    return MFREC_OK;
}

}  // namespace

extern "C" int mfrec_model_predict(mfrec_ctx *ctx, const mfrec_model *m, int predictor,
                                   const int32_t *pairs, const void *real, int real_is_f32, int64_t n,
                                   int is_device, double mu, double min_rating, double max_rating,
                                   double *out, double stats_out[4])
{
    if (!ctx || !m) return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_model_predict: NULL argument");
    if (predictor < 0 || predictor > MFREC_PRED_DOT)
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_model_predict: predictor=%d", predictor);
    if (n < 0 || (n > 0 && !pairs)) return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_model_predict: n=%lld", (long long)n);
    MF_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    if (n == 0) {
        if (stats_out) stats_out[0] = stats_out[1] = stats_out[2] = stats_out[3] = 0.0;
        return MFREC_OK;
    }
    DevBuf<int32_t> d_pairs, d_bad;
    DevBuf<char> d_real;
    DevBuf<double> d_out, d_part, d_stats;
    const size_t rsz = real_is_f32 ? 4 : 8;
    PredParams p;
    p.pairs = pairs;
    p.real = real;
    p.out = out;
    if (!is_device) {
        MF_CUDA(ctx, d_pairs.alloc((size_t)n * 2, ctx->stream));
        MF_CUDA(ctx, cudaMemcpyAsync(d_pairs.p, pairs, (size_t)n * 8, cudaMemcpyHostToDevice, st));
        p.pairs = d_pairs.p;
        if (real) {
            MF_CUDA(ctx, d_real.alloc((size_t)n * rsz, ctx->stream));
            MF_CUDA(ctx, cudaMemcpyAsync(d_real.p, real, (size_t)n * rsz, cudaMemcpyHostToDevice, st));
            p.real = d_real.p;
        }
        if (out) {
            MF_CUDA(ctx, d_out.alloc((size_t)n, ctx->stream));
            p.out = d_out.p;
        }
    }
    MF_CUDA(ctx, d_bad.alloc(1, ctx->stream));
    MF_CUDA(ctx, cudaMemsetAsync(d_bad.p, 0, 4, st));
    const int warps_per_block = 8;
    int grid = (int)std::min<int64_t>(ceil_div64(n, warps_per_block * 4), (int64_t)ctx->sm_count * 16);
    if (stats_out) {
        MF_CUDA(ctx, d_part.alloc((size_t)grid * 3, ctx->stream));
        MF_CUDA(ctx, d_stats.alloc(4, ctx->stream));
    }
    p.Q = m->Q; p.ib = m->ib; p.P = m->P; p.ub = m->ub;
    p.user_perm = m->user_perm; p.item_perm = m->item_perm;
    p.real_is_f32 = real_is_f32;
    p.n = n;
    p.predictor = predictor;
    p.mu = (float)mu; p.min_rating = (float)min_rating; p.max_rating = (float)max_rating;
    p.part = stats_out ? d_part.p : nullptr;
    p.ni = m->ni; p.nu = m->nu;
    p.bad = d_bad.p;
#define MF_PREDICT(E)                                                                                  \
    do {                                                                                               \
        if (m->p_kind == MFREC_STORAGE_F16) predict_kernel<E, __half><<<grid, 256, 0, st>>>(p);        \
        else if (m->p_kind == MFREC_STORAGE_BF16) predict_kernel<E, __nv_bfloat16><<<grid, 256, 0, st>>>(p); \
        else predict_kernel<E, float><<<grid, 256, 0, st>>>(p);                                        \
    } while (0)
    switch (m->kpad) {
    case 32: MF_PREDICT(1); break;
    case 64: MF_PREDICT(2); break;
    case 128: MF_PREDICT(4); break;
    case 256: MF_PREDICT(8); break;
    default: return mfrec_set_error(ctx, MFREC_ERR_UNSUPPORTED, "kpad=%d", m->kpad);
    }
#undef MF_PREDICT
    MF_LAUNCH_CHECK(ctx);
    if (stats_out) {
        stats_reduce_kernel<<<1, 256, 0, st>>>(d_part.p, grid, d_stats.p);
        MF_LAUNCH_CHECK(ctx);
        MF_CUDA(ctx, cudaMemcpyAsync(stats_out, d_stats.p, 32, cudaMemcpyDeviceToHost, st));
    }
    if (!is_device && out)
        MF_CUDA(ctx, cudaMemcpyAsync(out, d_out.p, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
    int32_t h_bad = 0;
    MF_CUDA(ctx, cudaMemcpyAsync(&h_bad, d_bad.p, 4, cudaMemcpyDeviceToHost, st));
    MF_CUDA(ctx, cudaStreamSynchronize(st));
    if (h_bad)
        return mfrec_set_error(ctx, MFREC_ERR_INDEX, "mfrec_model_predict: a pair has a user outside [0,%d) or an item outside [0,%d)",
                               m->nu, m->ni);
    return MFREC_OK;
}

namespace {

// A call that scores a handful of pairs (metrics.test_predict_rating's default is nbr_samples = 10)
// must not upload both factor matrices (0.5 GB at Netflix shape): gather the rows the pairs name
// into compact [k][m] arrays on the host and build a model of just those.
constexpr int64_t kSmallPairs = 4096;

struct CompactModel {
    std::vector<double> u, v, ib, ub;
    std::vector<int32_t> pairs;   // remapped to compact ids
    int32_t mi = 0, mu = 0;
};

// false: out of range index (the caller lets the full path report it)
bool gather_small(int k, const double *u, const double *v, int32_t ni, int32_t nu, const int32_t *pairs, int64_t n,
                  const double *items_bias, const double *users_bias, CompactModel &c)
{
    std::vector<int32_t> us(n), is(n);
    for (int64_t j = 0; j < n; ++j) {
        us[j] = pairs[2 * j];
        is[j] = pairs[2 * j + 1];
        if (us[j] < 0 || us[j] >= nu || is[j] < 0 || is[j] >= ni) return false;
    }
    std::vector<int32_t> uu(us), ii(is);
    std::sort(uu.begin(), uu.end());
    uu.erase(std::unique(uu.begin(), uu.end()), uu.end());
    std::sort(ii.begin(), ii.end());
    ii.erase(std::unique(ii.begin(), ii.end()), ii.end());
    c.mu = (int32_t)uu.size();
    c.mi = (int32_t)ii.size();
    c.u.resize((size_t)k * c.mi);
    c.v.resize((size_t)k * c.mu);
    for (int f = 0; f < k; ++f) {
        for (int32_t a = 0; a < c.mi; ++a) c.u[(size_t)f * c.mi + a] = u[(size_t)f * ni + ii[a]];
        for (int32_t a = 0; a < c.mu; ++a) c.v[(size_t)f * c.mu + a] = v[(size_t)f * nu + uu[a]];
    }
    if (items_bias) { c.ib.resize(c.mi); for (int32_t a = 0; a < c.mi; ++a) c.ib[a] = items_bias[ii[a]]; }
    if (users_bias) { c.ub.resize(c.mu); for (int32_t a = 0; a < c.mu; ++a) c.ub[a] = users_bias[uu[a]]; }
    c.pairs.resize((size_t)2 * n);
    for (int64_t j = 0; j < n; ++j) {
        c.pairs[2 * j] = (int32_t)(std::lower_bound(uu.begin(), uu.end(), us[j]) - uu.begin());
        c.pairs[2 * j + 1] = (int32_t)(std::lower_bound(ii.begin(), ii.end(), is[j]) - ii.begin());
    }
    return true;
}

// model for a one-shot call: compact when the pairs are few, the whole matrices otherwise
int model_for_pairs(mfrec_ctx *ctx, int k, const double *u, const double *v, int32_t ni, int32_t nu,
                    const int32_t *&pairs, int64_t n, const double *items_bias, const double *users_bias,
                    CompactModel &c, mfrec_model **M)
{
    if (n > 0 && n <= kSmallPairs && (int64_t)ni + nu > 8 * n && pairs &&
        gather_small(k, u, v, ni, nu, pairs, n, items_bias, users_bias, c)) {
        pairs = c.pairs.data();
        return mfrec_model_create(ctx, nullptr, k, c.mi, c.mu, c.u.data(), c.v.data(),
                                  items_bias ? c.ib.data() : nullptr, users_bias ? c.ub.data() : nullptr, M);
    }
    return mfrec_model_create(ctx, nullptr, k, ni, nu, u, v, items_bias, users_bias, M);
}

}  // namespace

extern "C" int mfrec_predict_pairs(mfrec_ctx *ctx, int predictor, int k, const double *u, const double *v,
                                   int32_t ni, int32_t nu, const int32_t *pairs, int64_t n, double mu,
                                   const double *items_bias, const double *users_bias,
                                   double min_rating, double max_rating, double *out)
{
    if (!ctx || !u || !v || !out) return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_predict_pairs: NULL argument");
    mfrec_model *M = nullptr;
    CompactModel compact;
    MF_TRY(model_for_pairs(ctx, k, u, v, ni, nu, pairs, n, items_bias, users_bias, compact, &M));
    const int rc = mfrec_model_predict(ctx, M, predictor, pairs, nullptr, 0, n, 0, mu, min_rating, max_rating, out, nullptr);
    mfrec_model_destroy(M);
    return rc;
}

extern "C" int mfrec_rmse_pairs(mfrec_ctx *ctx, int predictor, int k, const double *u, const double *v,
                                int32_t ni, int32_t nu, const int32_t *pairs, const double *real,
                                int64_t n, double mu, const double *items_bias, const double *users_bias,
                                double min_rating, double max_rating, double *errors_out, double stats[4])
{
    if (!ctx || !u || !v || !stats || (n > 0 && !real))
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_rmse_pairs: NULL argument");
    mfrec_model *M = nullptr;
    CompactModel compact;
    MF_TRY(model_for_pairs(ctx, k, u, v, ni, nu, pairs, n, items_bias, users_bias, compact, &M));
    double raw[4] = {0, 0, 0, 0};
    const int rc = mfrec_model_predict(ctx, M, predictor, pairs, real, 0, n, 0, mu, min_rating, max_rating,
                                       errors_out, raw);
    mfrec_model_destroy(M);
    if (rc != MFREC_OK) return rc;
    if (errors_out)
        for (int64_t j = 0; j < n; ++j) errors_out[j] = real[j] - errors_out[j];
    const double cnt = raw[2];
    if (cnt > 0) {
        const double mae = raw[1] / cnt, ms = raw[0] / cnt;
        stats[0] = sqrt(ms);
        stats[1] = mae;
        stats[2] = fmax(ms - mae * mae, 0.0);
        stats[3] = cnt;
    } else {
        stats[0] = stats[1] = stats[2] = NAN;
        stats[3] = 0.0;
    }
    return MFREC_OK;
}

extern "C" int mfrec_bias_stats(mfrec_ctx *ctx, const int32_t *ratings_index, const double *ratings,
                                int64_t nnz, int32_t ni, int32_t nu, double K2, double K3,
                                double *mu_out, double *items_bias, double *users_bias)
{
    if (!ctx || !mu_out || !items_bias || !users_bias || nnz < 0 || ni <= 0 || nu <= 0 ||
        (nnz > 0 && (!ratings_index || !ratings)))
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_bias_stats: bad argument");
    MF_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    if (nnz >= (1ll << 32)) return mfrec_set_error(ctx, MFREC_ERR_UNSUPPORTED, "mfrec_bias_stats: nnz >= 2^32");
    if (nnz == 0) {
        *mu_out = NAN;
        for (int32_t i = 0; i < ni; ++i) items_bias[i] = 0.0;
        for (int32_t j = 0; j < nu; ++j) users_bias[j] = 0.0;
        return MFREC_OK;
    }
    DevBuf<int32_t> d_idx, bad;
    DevBuf<double> d_r, acc_i, acc_u, part;
    const int grid = ctx->sm_count * 8;
    MF_CUDA(ctx, d_idx.alloc((size_t)nnz * 2, ctx->stream));
    MF_CUDA(ctx, d_r.alloc((size_t)nnz, ctx->stream));
    MF_CUDA(ctx, acc_i.alloc(ni, ctx->stream)); MF_CUDA(ctx, acc_u.alloc(nu, ctx->stream));
    MF_CUDA(ctx, part.alloc(grid, ctx->stream)); MF_CUDA(ctx, bad.alloc(1, ctx->stream));
    MF_TRY(mfrec_copy_h2d(ctx, d_idx.p, ratings_index, (size_t)nnz * 8, st));
    MF_TRY(mfrec_copy_h2d(ctx, d_r.p, ratings, (size_t)nnz * 8, st));
    MF_CUDA(ctx, cudaMemsetAsync(bad.p, 0, 4, st));
    sum_ratings_kernel<<<grid, 256, 0, st>>>(d_r.p, nnz, part.p);
    MF_LAUNCH_CHECK(ctx);
    std::vector<double> h_part(grid);
    MF_CUDA(ctx, cudaMemcpyAsync(h_part.data(), part.p, (size_t)grid * 8, cudaMemcpyDeviceToHost, st));
    MF_CUDA(ctx, cudaStreamSynchronize(st));
    double tot = 0.0;
    for (double x : h_part) tot += x;   // fixed grid, fixed order
    const double mu = tot / (double)nnz;
    MF_TRY(segmented_bias(ctx, d_idx.p, d_r.p, nnz, ni, nu, 0, mu, nullptr, K3, acc_i.p, bad.p));
    int32_t h_bad = 0;
    MF_CUDA(ctx, cudaMemcpyAsync(&h_bad, bad.p, 4, cudaMemcpyDeviceToHost, st));
    MF_CUDA(ctx, cudaStreamSynchronize(st));
    if (h_bad) return mfrec_set_error(ctx, MFREC_ERR_INDEX, "mfrec_bias_stats: index out of range");
    MF_TRY(segmented_bias(ctx, d_idx.p, d_r.p, nnz, ni, nu, 1, mu, acc_i.p, K2, acc_u.p, bad.p));
    MF_CUDA(ctx, cudaMemcpyAsync(items_bias, acc_i.p, (size_t)ni * 8, cudaMemcpyDeviceToHost, st));
    MF_CUDA(ctx, cudaMemcpyAsync(users_bias, acc_u.p, (size_t)nu * 8, cudaMemcpyDeviceToHost, st));
    MF_CUDA(ctx, cudaStreamSynchronize(st));
    *mu_out = mu;
    return MFREC_OK;
}

// predict_kernel scores each pair from its own two rows with the same per-lane order wherever the pair
// sits in the array (the four pairs of a warp iteration are reduced separately), so contiguous shares
// of the pairs give every pair the one-device result.
extern "C" int mfrec_model_predict_multi(mfrec_ctx *const *ctxs, const mfrec_model *const *models, int n_shards,
                                         int predictor, const int32_t *pairs, const void *real, int real_is_f32,
                                         int64_t n, double mu, double min_rating, double max_rating, double *out,
                                         double stats_out[4])
{
    const char *who = "mfrec_model_predict_multi";
    MF_TRY(mfrec_check_shards(ctxs, models, n_shards, who));
    if (predictor < 0 || predictor > MFREC_PRED_DOT)
        return mfrec_set_error(ctxs[0], MFREC_ERR_BAD_ARG, "%s: predictor=%d", who, predictor);
    if (n < 0 || (n > 0 && !pairs)) return mfrec_set_error(ctxs[0], MFREC_ERR_BAD_ARG, "%s: n=%lld", who, (long long)n);
    const size_t rsz = real_is_f32 ? 4 : 8;
    std::vector<double> st((size_t)n_shards * 4, 0.0);
    MF_TRY(mfrec_run_shards(ctxs, n_shards, who, [&](int s) -> int {
        const int64_t a = n * s / n_shards, b = n * (s + 1) / n_shards;
        if (a == b) return MFREC_OK;
        return mfrec_model_predict(ctxs[s], models[s], predictor, pairs + 2 * a,
                                   real ? static_cast<const char *>(real) + a * rsz : nullptr, real_is_f32, b - a, 0, mu,
                                   min_rating, max_rating, out ? out + a : nullptr, stats_out ? &st[(size_t)s * 4] : nullptr);
    }));
    if (stats_out)
        for (int j = 0; j < 4; ++j) {
            double acc = 0.0;
            for (int s = 0; s < n_shards; ++s) acc += st[(size_t)s * 4 + j];
            stats_out[j] = acc;
        }
    return MFREC_OK;
}
