// Funk-SVD per-feature SGD: estimator_loop_without_bias / _with_bias / _with_bias_dev of the
// reference (mfrec/lib/gd_estimator.pyx:691-779, 489-582, 588-685), as driven by
// GDRecommender.feature_training and retrain_user / retrain_item
// (mfrec/recommendation/gradient_descent.py:506-545, 879-905).
//
// One feature f is trained at a time: every rating touches ONE scalar of the item row and ONE of
// the user row plus a cached partial prediction, so a training pass is a pure stream:
//   12 B rating triple + 8 B cache read + 2 x (8 B read + 8 B write) scalars  (fp64 on device)
// Everything is kept in float64 with unfused multiplies and adds, so the stratified schedule is
// BIT-IDENTICAL to the CPU oracle replaying the same block order, and the sequential schedule is
// bit-identical to the reference order.
//
// Stratified schedule: the same B x B x W x W layout as the KMF kernel (pack.cu).  A warp owns a
// bucket and takes it 32 ratings at a time, one rating per lane (coalesced loads).  An update is
// scalar, so the only order that matters is between ratings that share a user or an item: the
// lanes compute the dependency LEVEL of their rating inside the batch (1 + the level of the latest
// earlier rating with the same user / the same item) and the batch runs level by level, all lanes
// of a level at once -- bit-identical to replaying the 32 ratings one after the other, in
// ~(number of levels) dependent updates instead of 32.  The item scalars of the column block and
// the user scalars of the row block live in shared memory.  The
// `while rmse <= rmse_last - min_improvement` control of the reference (rmse carried across
// features, max_epochs ignored) runs on the host, one device reduction per pass.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <numeric>

#include "common.cuh"
#include "fold.h"

namespace {

// gd_estimator.pyx:26-35 (`if x > 5: x = 5` then `if x < 1: x = 1`).  Both compares look at the
// incoming x, so they issue together: one float64 compare + selects on the hot item's serial
// chain instead of two compares back to back (same result for every x, NaN included).
__device__ __forceinline__ double clamp15(double x)
{
    const bool hi = x > 5.0, lo = x < 1.0;
    return hi ? 5.0 : (lo ? 1.0 : x);
}

// gd_estimator.pyx:38-73 with unfused arithmetic
__device__ __forceinline__ double funk_estimate(double uf, double vf, double cache, double base,
                                                double trail, int trailing)
{
    double s = cache > 0 ? cache : base;
    s = __dadd_rn(s, __dmul_rn(uf, vf));
    s = clamp15(s);
    if (trailing) {
        s = __dadd_rn(s, trail);
        s = clamp15(s);
    }
    return s;
}

// One rating of the reference loop (gd_estimator.pyx:588-685): the prediction from the cached
// partial prediction `cache` (or the baseline `base` while the cache is 0), the error, and the new
// item scalar (from the OLD mf, cf) handed to set_mf, then the new user scalar to set_cf, each only
// if its flag is set.  Returns the squared error.  funk_sequential_kernel and funk_fold_in_kernel
// share it, so both run the same operations in the same order.
template <class SetM, class SetC>
__device__ __forceinline__ double funk_rating(double r, double cache, double base, double trail, double lr,
                                              double K, double mf, double cf, int update_items,
                                              int update_users, SetM set_mf, SetC set_cf)
{
    const double pr = funk_estimate(mf, cf, cache, base, trail, 1);
    const double err = __dadd_rn(r, -pr);
    const double e2 = __dmul_rn(err, err);
    if (update_items) set_mf(__dadd_rn(mf, __dmul_rn(lr, __dadd_rn(__dmul_rn(err, cf), -__dmul_rn(K, mf)))));
    if (update_users) set_cf(__dadd_rn(cf, __dmul_rn(lr, __dadd_rn(__dmul_rn(err, mf), -__dmul_rn(K, cf)))));
    return e2;
}

struct FunkParams {
    const PackedRating *packed;
    const int64_t *bucket_off;
    const int32_t *bucket_cnt;
    const int32_t *col_start;
    const int32_t *row_start;   // [B*W + 1] first packed user id of every row group
    int user_rows;              // shared-memory slots for the user scalars of a row block
    double *uf;          // [ni] item scalars of feature f, packed order
    double *vf;          // [nu] user scalars
    const double *ibp;   // [ni] item biases, packed order (variant > 0)
    const double *ubp;   // [nu]
    const double *cache; // [packed_len]
    double *se_part;     // [B] per-CTA sums of this launch
    int32_t *ticks;      // [B] sub-epochs finished on each column block in this launch, or null
    int B, W, s_begin, s_end;
    int tile_rows;
    int variant;
    double lr, K, overall, trail;
    int update_users, update_items;
};

// One launch = sub-epochs [s_begin, s_end) of one training pass.  With `ticks` the launch is
// persistent and cooperative (all B sub-epochs): column blocks pass from CTA to CTA through
// release / acquire counters exactly as in sgd.cu, instead of one kernel boundary per sub-epoch,
// and inside a CTA column groups pass from warp to warp through shared-memory counters instead of
// a CTA-wide barrier per phase.
//
// A row block's user scalars stay in shared memory for the whole launch (8 bytes per user: 26 KB
// at Netflix shape), next to the column block's item scalars: the replay touches no global memory
// and needs none of the packer's stale-prefetch hints -- a re-read of a scalar that was just
// written is an ordinary shared-memory access one level later.  The next batch's ratings, cache
// values and biases are loaded while the current batch runs.
// (Round 2, profiles/r02m_funk_full.md: replaying the 32 ratings of a batch one after the other,
// every lane computing the same scalar update, was 57 warp instructions and ~360 cycles per
// rating: 5.3 ms per 20 M-rating pass.)
constexpr int kDeepDiv = 2;   // a batch with more than cnt / kDeepDiv levels is replayed serially

struct FunkStage {          // one staged rating of a deep batch, 32 bytes
    int u, i;               // user / item index relative to the row block / column block
    double r, c, b;         // rating, cached partial prediction, baseline
};

__global__ void __launch_bounds__(512) funk_train_kernel(const FunkParams prm)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int W = prm.W;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int rb = blockIdx.x;
    double *ufs = reinterpret_cast<double *>(smem_raw);
    double *ibs = ufs + prm.tile_rows;
    double *vfs = ibs + prm.tile_rows;
    double *se_s = vfs + prm.user_rows;
    FunkStage *stage_all = reinterpret_cast<FunkStage *>(se_s + W);
    int64_t *boff = reinterpret_cast<int64_t *>(stage_all + (size_t)W * 32);
    FunkStage *stage = stage_all + warp * 32;
    int32_t *bcnt = reinterpret_cast<int32_t *>(boff + W * W + 1);
    volatile int32_t *phase_done = reinterpret_cast<volatile int32_t *>(bcnt + ((W * W + 2) & ~1));
    const double lr = prm.lr, K = prm.K;
    double se = 0.0;
    // serial replay of the `cnt` ratings staged in stage[] (hot buckets and deep batches): every lane
    // computes the same update; the scalars of a run of equal items / equal users are forwarded in
    // registers, so a hot item's chain is ~10 dependent float64 operations per rating
    auto replay_staged = [&](int cnt, int &prev_u, int &prev_i, double &vf_cur, double &uf_cur, double &se_b) {
#pragma unroll 2
        for (int t = 0; t < cnt; ++t) {
            const FunkStage x = stage[t];   // broadcast loads
            const double cf = x.u == prev_u ? vf_cur : vfs[x.u];
            const double mf = x.i == prev_i ? uf_cur : ufs[x.i];
            const double pr = funk_estimate(mf, cf, x.c, x.b, prm.trail, 1);
            const double err = __dadd_rn(x.r, -pr);
            se_b = __dadd_rn(se_b, __dmul_rn(err, err));
            uf_cur = prm.update_items
                         ? __dadd_rn(mf, __dmul_rn(lr, __dadd_rn(__dmul_rn(err, cf), -__dmul_rn(K, mf))))
                         : mf;
            vf_cur = prm.update_users
                         ? __dadd_rn(cf, __dmul_rn(lr, __dadd_rn(__dmul_rn(err, mf), -__dmul_rn(K, cf))))
                         : cf;
            ufs[x.i] = uf_cur;     // every lane writes the same value
            vfs[x.u] = vf_cur;
            prev_u = x.u;
            prev_i = x.i;
        }
    };
    if (threadIdx.x < W) phase_done[threadIdx.x] = 0;
    // this row block's user scalars (no other CTA touches them during the launch)
    const int us0 = prm.row_start[rb * W], nub = prm.row_start[(rb + 1) * W] - us0;
    for (int i = threadIdx.x; i < nub; i += blockDim.x) vfs[i] = prm.vf[us0 + i];
    for (int s = prm.s_begin; s < prm.s_end; ++s) {
        const int step = s - prm.s_begin;
        const int cbl = (rb + s) % prm.B;
        const int cs = prm.col_start[cbl * W];
        const int nq = prm.col_start[(cbl + 1) * W] - cs;
        const int64_t bucket_base = ((int64_t)rb * prm.B + cbl) * W * W;
        for (int i = threadIdx.x; i <= W * W; i += blockDim.x) {
            boff[i] = prm.bucket_off[bucket_base + i];
            if (i < W * W) bcnt[i] = prm.bucket_cnt[bucket_base + i];
        }
        if (prm.ticks && threadIdx.x == 0)
            while (ld_acquire_gpu(prm.ticks + cbl) < s) __nanosleep(64);
        __syncthreads();   // the column block is ours; descriptors (and, first time, vfs) visible
        // item scalars: L2 loads (another SM wrote them; L1 may hold a stale line)
        for (int i = threadIdx.x; i < nq; i += blockDim.x) {
            ufs[i] = __ldcg(prm.uf + cs + i);
            ibs[i] = prm.variant ? prm.ibp[cs + i] : 0.0;
        }
        __syncthreads();
        const int32_t done_base = step * W;
        for (int p = 0; p < W; ++p) {
            const int64_t a = boff[warp * W + p];
            const int n = bcnt[warp * W + p];
            // first batch: triple, cache value, user bias (nothing of this is written by the pass)
            PackedRating rt;
            rt.u = us0; rt.i = cs; rt.r = 0.f;
            double c = 0.0, ubv = 0.0;
            if (lane < n) {
                rt = prm.packed[a + lane];
                c = prm.cache[a + lane];
                if (prm.variant) ubv = prm.ubp[rt.u & kIdMask];
            }
            if (p > 0) {
                // column group (warp + p) mod W comes from warp + 1, which used it in phase p - 1
                const volatile int32_t *flag = phase_done + (warp + 1 == W ? 0 : warp + 1);
                if (lane == 0) {
                    while (*flag < done_base + p) __nanosleep(32);
                    __threadfence_block();
                }
                __syncwarp();
            }
            // A hot item's bucket (most of its first 32 ratings on the item of the first or of the last
            // one) is ONE chain, and the hottest item's chain bounds the pass: replay it rating by
            // rating, every lane computing the same update, the scalars of a run of equal items /
            // equal users forwarded in registers across the whole bucket -- ~10 dependent float64
            // operations per rating and nothing else on the chain.
            bool hot_bucket = false;
            if (n >= 16) {
                const int c0 = min(32, n), il0 = (rt.i & kIdMask) - cs;
                const int i_first = __shfl_sync(0xffffffffu, il0, 0), i_last = __shfl_sync(0xffffffffu, il0, c0 - 1);
                hot_bucket = kDeepDiv * max(__popc(__ballot_sync(0xffffffffu, lane < c0 && il0 == i_first)),
                                            __popc(__ballot_sync(0xffffffffu, lane < c0 && il0 == i_last))) > c0;
            }
            if (hot_bucket) {
                int prev_u = -1, prev_i = -1;
                double vf_cur = 0.0, uf_cur = 0.0, se_b = 0.0;
                for (int base = 0; base < n; base += 32) {
                    const int cnt = min(32, n - base);
                    __syncwarp();   // the previous batch has been replayed by every lane
                    {
                        const int il = (rt.i & kIdMask) - cs;
                        FunkStage st;
                        st.u = (rt.u & kIdMask) - us0; st.i = il; st.r = (double)rt.r; st.c = c;
                        // variant 0 uses the estimator's defaults: overall 1.0, biases 0 (:751)
                        st.b = prm.variant ? __dadd_rn(__dadd_rn(prm.overall, ibs[il]), ubv) : 1.0;
                        stage[lane] = st;
                    }
                    {   // next batch's inputs, in flight during the replay
                        const int j = base + 32 + lane;
                        rt.u = us0; rt.i = cs; rt.r = 0.f;
                        c = 0.0; ubv = 0.0;
                        if (j < n) {
                            rt = prm.packed[a + j];
                            c = prm.cache[a + j];
                            if (prm.variant) ubv = prm.ubp[rt.u & kIdMask];
                        }
                    }
                    __syncwarp();
                    replay_staged(cnt, prev_u, prev_i, vf_cur, uf_cur, se_b);
                }
                if (lane == 0) se = __dadd_rn(se, se_b);
                __syncwarp();
            } else
            for (int base = 0; base < n; base += 32) {
                const int cnt = min(32, n - base);
                // this lane's rating of the batch (loaded one batch ahead)
                const bool live = lane < cnt;
                const int ul = (rt.u & kIdMask) - us0, il = (rt.i & kIdMask) - cs;
                const double r = (double)rt.r, cc = c;
                // variant 0 uses the estimator's defaults: overall 1.0, biases 0 (:751)
                const double bb = prm.variant ? __dadd_rn(__dadd_rn(prm.overall, ibs[il]), ubv) : 1.0;
                // next batch's inputs, in flight while this one is replayed
                {
                    const int j = base + 32 + lane;
                    rt.u = us0; rt.i = cs; rt.r = 0.f;
                    c = 0.0; ubv = 0.0;
                    if (j < n) {
                        rt = prm.packed[a + j];
                        c = prm.cache[a + j];
                        if (prm.variant) ubv = prm.ubp[rt.u & kIdMask];
                    }
                }
                // Dependency levels: a rating depends on the latest earlier rating of the batch with
                // the same user or the same item.  level = 1 + max(level of those two) (longest path,
                // relaxed until nothing changes: as many rounds as there are levels).  Ratings of one
                // level share no scalar, so the lanes of a level run together; levels run in order.
                const unsigned below = (1u << lane) - 1u;
                bool deep;
                int pu = -1, pi = -1;
                {
                    // the packer orders a bucket by (user, item): equal users are neighbours
                    const int u_prev = __shfl_up_sync(0xffffffffu, ul, 1);
                    const bool sorted = !__any_sync(0xffffffffu, live && lane > 0 && ul < u_prev);
                    if (sorted) {
                        pu = (live && lane > 0 && ul == u_prev) ? lane - 1 : -1;
                    } else {
                        pu = 31 - __clz(__match_any_sync(0xffffffffu, live ? ul : -1 - lane) & below);   // -1: none
                    }
                    const unsigned same_i = __match_any_sync(0xffffffffu, live ? il : -1 - lane);
                    pi = 31 - __clz(same_i & below);
                    deep = kDeepDiv * __reduce_max_sync(0xffffffffu, __popc(same_i)) > cnt;
                }
                int level = 1;
                for (int round = 1; !deep; ++round) {
                    const int lu = __shfl_sync(0xffffffffu, level, pu < 0 ? lane : pu);
                    const int li = __shfl_sync(0xffffffffu, level, pi < 0 ? lane : pi);
                    int nl = 1;
                    if (pu >= 0) nl = lu + 1;
                    if (pi >= 0) nl = max(nl, li + 1);
                    const bool changed = nl != level;
                    level = nl;
                    if (!__any_sync(0xffffffffu, changed)) break;
                    deep = kDeepDiv * round >= cnt;   // some rating sits at level round + 1 or deeper
                }
                const int lmax = deep ? 0 : __reduce_max_sync(0xffffffffu, live ? level : 0);
                if (deep) {
                    // A deep batch (the ratings of a hot item: one chain): replay it rating by rating,
                    // every lane computing the same update, the scalars of a run of equal items / equal
                    // users forwarded in registers -- ~10 dependent float64 operations per rating and
                    // no shared-memory round trip on the chain.
                    FunkStage st;
                    st.u = ul; st.i = il; st.r = r; st.c = cc; st.b = bb;
                    stage[lane] = st;
                    __syncwarp();
                    int prev_u = -1, prev_i = -1;
                    double vf_cur = 0.0, uf_cur = 0.0, se_b = 0.0;
                    replay_staged(cnt, prev_u, prev_i, vf_cur, uf_cur, se_b);
                    if (lane == 0) se = __dadd_rn(se, se_b);
                    __syncwarp();   // the batch has been replayed by every lane (stage may be refilled)
                    continue;
                }
                for (int L = 1; L <= lmax; ++L) {
                    if (live && level == L) {
                        const double cf = vfs[ul];
                        const double mf = ufs[il];
                        const double pr = funk_estimate(mf, cf, cc, bb, prm.trail, 1);
                        const double err = __dadd_rn(r, -pr);
                        se = __dadd_rn(se, __dmul_rn(err, err));
                        if (prm.update_items)
                            ufs[il] = __dadd_rn(mf, __dmul_rn(lr, __dadd_rn(__dmul_rn(err, cf), -__dmul_rn(K, mf))));
                        if (prm.update_users)
                            vfs[ul] = __dadd_rn(cf, __dmul_rn(lr, __dadd_rn(__dmul_rn(err, mf), -__dmul_rn(K, cf))));
                    }
                    __syncwarp();   // the level's stores are visible to the next level's lanes
                }
            }
            // hand the column group over: item scalars written above, then the counter
            __syncwarp();
            if (lane == 0) {
                __threadfence_block();
                phase_done[warp] = done_base + p + 1;
            }
        }
        __syncthreads();   // every warp is done with the tile
        for (int i = threadIdx.x; i < nq; i += blockDim.x) prm.uf[cs + i] = ufs[i];
        if (prm.ticks) {
            __threadfence();
            __syncthreads();
            if (threadIdx.x == 0) st_release_gpu(prm.ticks + cbl, s + 1);
        } else {
            __syncthreads();
        }
    }
    for (int i = threadIdx.x; i < nub; i += blockDim.x) prm.vf[us0 + i] = vfs[i];
    // every lane holds the squared errors of its own ratings: fixed-order (deterministic) reduction
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) se = __dadd_rn(se, __shfl_xor_sync(0xffffffffu, se, o));
    if (lane == 0) se_s[warp] = se;
    __syncthreads();
    if (threadIdx.x == 0) {
        double tot = 0.0;
        for (int w = 0; w < W; ++w) tot = __dadd_rn(tot, se_s[w]);
        prm.se_part[rb] = tot;
    }
}

// cache refresh after a feature is trained (:771-777): embarrassingly parallel
__global__ void funk_cache_kernel(const PackedRating *__restrict__ packed, int64_t n,
                                  const double *__restrict__ uf, const double *__restrict__ vf,
                                  const double *__restrict__ ibp, const double *__restrict__ ubp,
                                  int variant, double overall, double *__restrict__ cache)
{
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += stride) {
        PackedRating rt = packed[j];
        if (rt.i & kFlagPad) continue;
        rt.u &= kIdMask;
        rt.i &= kIdMask;
        const double bb = variant ? __dadd_rn(__dadd_rn(overall, ibp[rt.i]), ubp[rt.u]) : 1.0;
        cache[j] = funk_estimate(uf[rt.i], vf[rt.u], cache[j], bb, 0.0, 0);
    }
}

__global__ void gather_row_kernel(const double *__restrict__ row, int32_t n,
                                  const int32_t *__restrict__ perm, double *__restrict__ out)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[perm[i]] = row ? row[i] : 0.0;
}

__global__ void scatter_row_kernel(const double *__restrict__ in, int32_t n,
                                   const int32_t *__restrict__ perm, double *__restrict__ row)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) row[i] = in[perm[i]];
}

__global__ void __launch_bounds__(1024) sum_parts_kernel(const double *__restrict__ part, int n,
                                                         double *__restrict__ out)
{
    // fixed order: one thread, partials are few (B * B per pass)
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        double tot = 0.0;
        for (int i = 0; i < n; ++i) tot = __dadd_rn(tot, part[i]);
        *out = tot;
    }
}

// ---- sequential schedule: the reference loop in the reference's order --------------------------
// One warp, 32 ratings of the stream at a time, one rating per lane, run by dependency level
// inside the window (see funk_train_kernel): bit-identical to one thread walking the stream.  The
// squared errors are summed in stream order -- the sum decides `rmse <= rmse_last - min_improvement`.
__global__ void __launch_bounds__(32)
funk_sequential_kernel(int variant, int min_epochs, double min_improvement, int dim,
                       double f_init, double lr, double K, double overall,
                       double *u, double *v, const int32_t *idx, const double *ratings,
                       int64_t nnz, int64_t ni, int64_t nu, const double *ib,
                       const double *ub, int update_users, int update_items,
                       double *cache, int32_t *feature_epochs, double *feature_rmse)
{
    if (blockIdx.x != 0) return;
    const int lane = threadIdx.x;
    const unsigned FULLM = 0xffffffffu;
    double rmse = 2.0, rmse_last = 0.0;
    for (int64_t n = lane; n < nnz; n += 32) cache[n] = 0.0;
    __syncwarp();
    for (int f = 0; f < dim; ++f) {
        double *uf = u + (int64_t)f * ni, *vf = v + (int64_t)f * nu;
        const double trail = __dmul_rn(__dmul_rn((double)(dim - f - 1), f_init), f_init);
        int epoch = 0;
        while (epoch < min_epochs || rmse <= __dadd_rn(rmse_last, -min_improvement)) {   // (warp-uniform)
            double se = 0.0;
            rmse_last = rmse;
            for (int64_t base = 0; base < nnz; base += 32) {
                const int cnt = (int)(nnz - base < 32 ? nnz - base : 32);
                const bool live = lane < cnt;
                const int64_t n = base + lane;
                int user = 0, item = 0;
                double r = 0.0, cc = 0.0, bb = 1.0;
                if (live) {
                    user = idx[2 * n]; item = idx[2 * n + 1];
                    r = ratings[n]; cc = cache[n];
                    if (variant) bb = __dadd_rn(__dadd_rn(overall, ib[item]), ub[user]);
                }
                int lmax;
                const int level = mfrec_window_levels(user, item, live, lane, lmax);   // common.cuh
                double e2 = 0.0;
                for (int L = 1; L <= lmax; ++L) {
                    if (live && level == L) {
                        const double cf = vf[user], mf = uf[item];
                        e2 = funk_rating(r, cc, bb, trail, lr, K, mf, cf, update_items, update_users,
                                         [&](double x) { uf[item] = x; }, [&](double x) { vf[user] = x; });
                    }
                    __syncwarp();   // this level's stores are visible to the lanes of the next
                }
                for (int t = 0; t < cnt; ++t) se = __dadd_rn(se, __shfl_sync(FULLM, e2, t));   // stream order
            }
            rmse = sqrt(se / (double)nnz);
            ++epoch;
        }
        if (lane == 0) {
            feature_epochs[f] = epoch;
            feature_rmse[f] = rmse;
        }
        for (int64_t n = lane; n < nnz; n += 32) {
            const int user = idx[2 * n], item = idx[2 * n + 1];
            const double bb = variant ? __dadd_rn(__dadd_rn(overall, ib[item]), ub[user]) : 1.0;
            cache[n] = funk_estimate(uf[item], vf[user], cache[n], bb, 0.0, 0);
        }
        __syncwarp();
    }
}

// ---- batched fold-in (mfrec_fold_in_funk) -------------------------------------------------------
// Many fold-ins of the kind GDRecommender.retrain_user / retrain_item make (gradient_descent.py:
// 879-905): each trains ONE row on its own ratings with estimator_loop_with_bias_dev, the other side
// frozen by the update flags.  That loop reads both bias arrays and the frozen side and writes
// nothing but the row, so two fold-ins share no written state: all rows run in one launch, ONE LANE
// PER ROW, in any order.
//
// A lane replays funk_sequential_kernel for its row.  Every rating names the row, so each one
// depends on the one before it: the lane walks them in input order through funk_rating and sums the
// squared errors in that order.  Within feature f the row's scalar t stays in a register, and what
// else a rating's update reads is constant: the frozen scalar o and s0 = cache > 0 ? cache : base.
// Both are staged once per feature (so[], ss[]) and loaded kAhead ratings ahead of the update that
// needs them, so the chain is the ~13 dependent float64 operations of the update and no memory
// round trip.  The cache refresh after a feature is folded into the next feature's staging.
//
// Jobs (rows) are sorted by rating count, longest first; block w holds jobs [32w, 32w + 32).  The
// per-rating arrays are warp-interleaved: rating n of lane l of block w sits at
// warp_off[w] + 32 n + l, so the lanes of a warp load consecutive addresses.  trained / frozen are
// compact row-major [m][dim]; tbias / fbias their biases; fidx the frozen row of every rating.
constexpr int kAhead = 8;   // ratings whose staged inputs are in flight ahead of the update

template <int SIDE>
__global__ void __launch_bounds__(32)
funk_fold_in_kernel(int min_epochs, double min_improvement, int dim, double f_init, double lr, double K,
                    double overall, double *__restrict__ trained, const double *__restrict__ tbias,
                    const double *__restrict__ frozen, const double *__restrict__ fbias,
                    const int32_t *__restrict__ job_row, const int32_t *__restrict__ job_cnt,
                    const int64_t *__restrict__ warp_off, const int32_t *__restrict__ fidx,
                    const double *__restrict__ rv, double *__restrict__ base, double *__restrict__ so,
                    double *__restrict__ ss, int32_t n_jobs, int32_t *__restrict__ feature_epochs,
                    double *__restrict__ feature_rmse)
{
    const int32_t j = blockIdx.x * 32 + threadIdx.x;
    if (j >= n_jobs) return;
    const int32_t row = job_row[j], cnt = job_cnt[j];
    const int64_t p0 = warp_off[blockIdx.x] + threadIdx.x;
    double *const grow = trained + (size_t)row * dim;
    // the baseline of every rating: overall + b_item + b_user, in that order (gd_estimator.pyx:38-73)
    const double tb = tbias[row];
    for (int n = 0; n < cnt; ++n) {
        const int64_t p = p0 + 32 * (int64_t)n;
        const double fb = fbias[fidx[p]];
        base[p] = SIDE == MFREC_FOLD_USERS ? __dadd_rn(__dadd_rn(overall, fb), tb)
                                           : __dadd_rn(__dadd_rn(overall, tb), fb);
    }
    // rating n's staged inputs, or nothing past the row's end
    auto load = [&](int n, double &o, double &s, double &r) {
        if (n < cnt) {
            const int64_t p = p0 + 32 * (int64_t)n;
            o = so[p]; s = ss[p]; r = rv[p];
        } else {
            o = 0.0; s = 0.0; r = 0.0;
        }
    };
    double rmse = 2.0, rmse_last = 0.0, t = 0.0;
    for (int f = 0; f < dim; ++f) {
        // stage feature f: the frozen scalars, and s0 from the cache feature f - 1 left behind
        // (funk_sequential_kernel's refresh: funk_estimate(..., trailing = 0); the cache is 0 at f = 0)
        for (int n = 0; n < cnt; ++n) {
            const int64_t p = p0 + 32 * (int64_t)n;
            double s0 = base[p];
            if (f > 0) {
                const double o = so[p], sp = ss[p];
                const double c = SIDE == MFREC_FOLD_USERS ? funk_estimate(o, t, sp, sp, 0.0, 0)
                                                          : funk_estimate(t, o, sp, sp, 0.0, 0);
                s0 = c > 0 ? c : s0;
            }
            ss[p] = s0;
            so[p] = frozen[(size_t)fidx[p] * dim + f];
        }
        t = grow[f];
        const double trail = __dmul_rn(__dmul_rn((double)(dim - f - 1), f_init), f_init);
        int epoch = 0;
        while (epoch < min_epochs || rmse <= __dadd_rn(rmse_last, -min_improvement)) {
            double se = 0.0;
            rmse_last = rmse;
            double o[kAhead], s[kAhead], r[kAhead];
#pragma unroll
            for (int i = 0; i < kAhead; ++i) load(i, o[i], s[i], r[i]);
            for (int n0 = 0; n0 < cnt; n0 += kAhead) {
                double on[kAhead], sn[kAhead], rn[kAhead];
#pragma unroll
                for (int i = 0; i < kAhead; ++i) load(n0 + kAhead + i, on[i], sn[i], rn[i]);
#pragma unroll
                for (int i = 0; i < kAhead; ++i) {
                    if (n0 + i < cnt) {
                        const auto set_t = [&](double x) { t = x; };
                        const auto frozen_side = [](double) {};
                        const double e2 = SIDE == MFREC_FOLD_USERS
                            ? funk_rating(r[i], s[i], s[i], trail, lr, K, o[i], t, 0, 1, frozen_side, set_t)
                            : funk_rating(r[i], s[i], s[i], trail, lr, K, t, o[i], 1, 0, set_t, frozen_side);
                        se = __dadd_rn(se, e2);
                    }
                    o[i] = on[i]; s[i] = sn[i]; r[i] = rn[i];
                }
            }
            rmse = sqrt(se / (double)cnt);
            ++epoch;
        }
        grow[f] = t;
        feature_epochs[(size_t)j * dim + f] = epoch;
        feature_rmse[(size_t)j * dim + f] = rmse;
    }
}

size_t funk_smem_bytes(int tile_rows, int user_rows, int W)
{
    return (size_t)tile_rows * 16 + (size_t)user_rows * 8 + (size_t)W * 8 + (size_t)W * 32 * sizeof(FunkStage) +
           (size_t)(W * W + 1) * 8 + (size_t)(W * W + 4) * 4 + (size_t)(W + 4) * 4 + 64;
}

}  // namespace

extern "C" int mfrec_train_funk(mfrec_ctx *ctx, int variant, int min_epochs, int max_epochs,
                                double min_improvement, int k, double f_init, double learning_rate,
                                double K, double overall_avg, double *u, double *v,
                                const int32_t *ratings_index, const double *ratings, int64_t nnz,
                                int32_t ni, int32_t nu, const double *items_bias,
                                const double *users_bias, int update_users, int update_items,
                                const mfrec_opts *opts, int32_t *feature_epochs, double *feature_rmse)
{
    (void)max_epochs;  // ignored by the reference too (CYTHON_UNUSED, gd_estimator.c:1272)
    if (!ctx) return mfrec_set_error(nullptr, MFREC_ERR_BAD_ARG, "mfrec_train_funk: NULL ctx");
    if (variant < MFREC_FUNK_WITHOUT_BIAS || variant > MFREC_FUNK_WITH_BIAS_DEV)
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_train_funk: variant=%d", variant);
    if (!u || !v || (nnz > 0 && (!ratings_index || !ratings)) || k <= 0 || ni <= 0 || nu <= 0 || nnz < 0)
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_train_funk: bad argument");
    if (variant != MFREC_FUNK_WITHOUT_BIAS && (!items_bias || !users_bias))
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_train_funk: bias arrays are required");
    if (variant != MFREC_FUNK_WITH_BIAS_DEV) { update_users = 1; update_items = 1; }
    if (nnz == 0)
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG,
                               "mfrec_train_funk: no ratings (the reference loops forever on 0/0)");
    MF_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    std::vector<int32_t> h_fe(k, 0);
    std::vector<double> h_fr(k, 0.0);

    DevBuf<double> du, dv, dib, dub;
    MF_CUDA(ctx, du.alloc((size_t)k * ni, ctx->stream));
    MF_CUDA(ctx, dv.alloc((size_t)k * nu, ctx->stream));
    MF_CUDA(ctx, cudaMemcpyAsync(du.p, u, (size_t)k * ni * 8, cudaMemcpyHostToDevice, st));
    MF_CUDA(ctx, cudaMemcpyAsync(dv.p, v, (size_t)k * nu * 8, cudaMemcpyHostToDevice, st));
    if (variant) {
        MF_CUDA(ctx, dib.alloc(ni, ctx->stream));
        MF_CUDA(ctx, dub.alloc(nu, ctx->stream));
        MF_CUDA(ctx, cudaMemcpyAsync(dib.p, items_bias, (size_t)ni * 8, cudaMemcpyHostToDevice, st));
        MF_CUDA(ctx, cudaMemcpyAsync(dub.p, users_bias, (size_t)nu * 8, cudaMemcpyHostToDevice, st));
    }

    if (opts && opts->schedule == MFREC_SCHED_SEQUENTIAL) {
        for (int64_t n = 0; n < nnz; ++n) {
            const int32_t a = ratings_index[2 * n], b = ratings_index[2 * n + 1];
            if (a < 0 || a >= nu || b < 0 || b >= ni)
                return mfrec_set_error(ctx, MFREC_ERR_INDEX, "mfrec_train_funk: rating %lld has (user,item)=(%d,%d)",
                                       (long long)n, a, b);
        }
        DevBuf<int32_t> didx, dfe;
        DevBuf<double> dr, dcache, dfr;
        MF_CUDA(ctx, didx.alloc((size_t)nnz * 2, ctx->stream));
        MF_CUDA(ctx, dr.alloc(nnz, ctx->stream));
        MF_CUDA(ctx, dcache.alloc(nnz, ctx->stream));
        MF_CUDA(ctx, dfe.alloc(k, ctx->stream));
        MF_CUDA(ctx, dfr.alloc(k, ctx->stream));
        MF_CUDA(ctx, cudaMemcpyAsync(didx.p, ratings_index, (size_t)nnz * 8, cudaMemcpyHostToDevice, st));
        MF_CUDA(ctx, cudaMemcpyAsync(dr.p, ratings, (size_t)nnz * 8, cudaMemcpyHostToDevice, st));
        funk_sequential_kernel<<<1, 32, 0, st>>>(variant, min_epochs, min_improvement, k, f_init,
                                                learning_rate, K, overall_avg, du.p, dv.p, didx.p, dr.p,
                                                nnz, ni, nu, dib.p, dub.p, update_users, update_items,
                                                dcache.p, dfe.p, dfr.p);
        MF_LAUNCH_CHECK(ctx);
        MF_CUDA(ctx, cudaMemcpyAsync(h_fe.data(), dfe.p, (size_t)k * 4, cudaMemcpyDeviceToHost, st));
        MF_CUDA(ctx, cudaMemcpyAsync(h_fr.data(), dfr.p, (size_t)k * 8, cudaMemcpyDeviceToHost, st));
    } else {
        mfrec_opts o;
        if (opts) o = *opts; else memset(&o, 0, sizeof(o));
        o.n_slabs = 1;
        o.split = MFREC_SPLIT_OFF;   // bit-exact with the reference order: no item copies here
        o.k_hint = 4;   // the tile holds 16 B per item here, far below any factor-row tile
        mfrec_ratings *R = nullptr;
        MF_TRY(mfrec_ratings_pack(ctx, ratings_index, ratings, 0, 0, nnz, ni, nu, nullptr, &o, &R));
        struct Guard { mfrec_ratings *r; ~Guard() { mfrec_ratings_destroy(r); } } guard{R};
        // user scalars of a row block live in shared memory: widest row block (users)
        int user_rows = 0;
        for (int b = 0; b < R->B; ++b)
            user_rows = std::max(user_rows, R->h_row_start[(size_t)(b + 1) * R->W] - R->h_row_start[(size_t)b * R->W]);
        user_rows = (user_rows + 1) & ~1;
        const size_t smem = funk_smem_bytes(R->max_cb_items, user_rows, R->W);
        if (smem > ctx->smem_optin)
            return mfrec_set_error(ctx, MFREC_ERR_UNSUPPORTED,
                                   "mfrec_train_funk: %d item and %d user scalars per block need %zu B shared memory (> %zu)",
                                   R->max_cb_items, user_rows, smem, ctx->smem_optin);
        DevBuf<int32_t> row_start;
        MF_CUDA(ctx, row_start.alloc(R->h_row_start.size(), ctx->stream));
        MF_CUDA(ctx, cudaMemcpyAsync(row_start.p, R->h_row_start.data(), R->h_row_start.size() * 4,
                                     cudaMemcpyHostToDevice, st));
        MF_CUDA(ctx, cudaFuncSetAttribute(funk_train_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        DevBuf<double> cache, ufp, vfp, ibp, ubp, se_part, se_tot;
        MF_CUDA(ctx, cache.alloc((size_t)R->packed_len + 1, ctx->stream));
        MF_CUDA(ctx, cudaMemsetAsync(cache.p, 0, ((size_t)R->packed_len + 1) * 8, st));
        MF_CUDA(ctx, ufp.alloc(ni, ctx->stream));
        MF_CUDA(ctx, vfp.alloc(nu, ctx->stream));
        MF_CUDA(ctx, ibp.alloc(ni, ctx->stream));
        MF_CUDA(ctx, ubp.alloc(nu, ctx->stream));
        MF_CUDA(ctx, se_part.alloc((size_t)R->B * R->B, ctx->stream));
        // one persistent cooperative launch per pass when all B CTAs fit at once (see sgd.cu)
        const bool persistent = ctx->coop_launch && !getenv("MFREC_SGD_LAUNCH_PER_SUBEPOCH") && R->B <= ctx->sm_count;
        DevBuf<int32_t> ticks;
        MF_CUDA(ctx, ticks.alloc(R->B, ctx->stream));
        MF_CUDA(ctx, se_tot.alloc(1, ctx->stream));
        const int gi = (ni + 255) / 256, gu = (nu + 255) / 256;
        gather_row_kernel<<<gi, 256, 0, st>>>(variant ? dib.p : nullptr, ni, R->item_perm, ibp.p);
        MF_LAUNCH_CHECK(ctx);
        gather_row_kernel<<<gu, 256, 0, st>>>(variant ? dub.p : nullptr, nu, R->user_perm, ubp.p);
        MF_LAUNCH_CHECK(ctx);
        FunkParams prm;
        prm.packed = R->packed; prm.bucket_off = R->bucket_off; prm.bucket_cnt = R->bucket_cnt;
        prm.col_start = R->col_start;
        prm.row_start = row_start.p;
        prm.user_rows = user_rows;
        prm.uf = ufp.p; prm.vf = vfp.p; prm.ibp = ibp.p; prm.ubp = ubp.p; prm.cache = cache.p;
        prm.B = R->B; prm.W = R->W; prm.tile_rows = R->max_cb_items; prm.variant = variant;
        prm.lr = learning_rate; prm.K = K; prm.overall = overall_avg;
        prm.update_users = update_users; prm.update_items = update_items;
        double rmse = 2.0, rmse_last = 0.0;
        for (int f = 0; f < k; ++f) {
            gather_row_kernel<<<gi, 256, 0, st>>>(du.p + (size_t)f * ni, ni, R->item_perm, ufp.p);
            MF_LAUNCH_CHECK(ctx);
            gather_row_kernel<<<gu, 256, 0, st>>>(dv.p + (size_t)f * nu, nu, R->user_perm, vfp.p);
            MF_LAUNCH_CHECK(ctx);
            prm.trail = (double)(k - f - 1) * f_init * f_init;
            int epoch = 0;
            while (epoch < min_epochs || rmse <= rmse_last - min_improvement) {
                rmse_last = rmse;
                if (persistent) {
                    MF_CUDA(ctx, cudaMemsetAsync(ticks.p, 0, (size_t)R->B * 4, st));
                    prm.s_begin = 0; prm.s_end = R->B; prm.ticks = ticks.p; prm.se_part = se_part.p;
                    void *args[] = {(void *)&prm};
                    MF_CUDA(ctx, cudaLaunchCooperativeKernel((const void *)funk_train_kernel, dim3(R->B), dim3(R->W * 32),
                                                             args, smem, st));
                    ctx->launches += 1;
                } else {
                    for (int s = 0; s < R->B; ++s) {
                        prm.s_begin = s; prm.s_end = s + 1; prm.ticks = nullptr;
                        prm.se_part = se_part.p + (size_t)s * R->B;
                        funk_train_kernel<<<R->B, R->W * 32, smem, st>>>(prm);
                        MF_LAUNCH_CHECK(ctx);
                    }
                }
                sum_parts_kernel<<<1, 32, 0, st>>>(se_part.p, persistent ? R->B : R->B * R->B, se_tot.p);
                MF_LAUNCH_CHECK(ctx);
                double se = 0.0;
                MF_CUDA(ctx, cudaMemcpyAsync(&se, se_tot.p, 8, cudaMemcpyDeviceToHost, st));
                MF_CUDA(ctx, cudaStreamSynchronize(st));
                rmse = sqrt(se / (double)nnz);
                ++epoch;
            }
            h_fe[f] = epoch;
            h_fr[f] = rmse;
            funk_cache_kernel<<<ctx->sm_count * 8, 256, 0, st>>>(R->packed, R->packed_len, ufp.p, vfp.p,
                                                                 ibp.p, ubp.p, variant, overall_avg, cache.p);
            MF_LAUNCH_CHECK(ctx);
            scatter_row_kernel<<<gi, 256, 0, st>>>(ufp.p, ni, R->item_perm, du.p + (size_t)f * ni);
            MF_LAUNCH_CHECK(ctx);
            scatter_row_kernel<<<gu, 256, 0, st>>>(vfp.p, nu, R->user_perm, dv.p + (size_t)f * nu);
            MF_LAUNCH_CHECK(ctx);
        }
        MF_CUDA(ctx, cudaStreamSynchronize(st));
    }
    MF_CUDA(ctx, cudaMemcpyAsync(u, du.p, (size_t)k * ni * 8, cudaMemcpyDeviceToHost, st));
    MF_CUDA(ctx, cudaMemcpyAsync(v, dv.p, (size_t)k * nu * 8, cudaMemcpyDeviceToHost, st));
    MF_CUDA(ctx, cudaStreamSynchronize(st));
    if (feature_epochs) memcpy(feature_epochs, h_fe.data(), (size_t)k * 4);
    if (feature_rmse) memcpy(feature_rmse, h_fr.data(), (size_t)k * 8);
    return MFREC_OK;
}

extern "C" int mfrec_fold_in_funk(mfrec_ctx *ctx, int side, int min_epochs, double min_improvement, int k,
                                  double f_init, double learning_rate, double K, double overall_avg,
                                  double *u, double *v, const int32_t *ratings_index, const double *ratings,
                                  int64_t nnz, int32_t ni, int32_t nu, const double *items_bias,
                                  const double *users_bias, const int32_t *rows, int32_t n_rows,
                                  int32_t *feature_epochs, double *feature_rmse)
{
    if (!ctx) return mfrec_set_error(nullptr, MFREC_ERR_BAD_ARG, "mfrec_fold_in_funk: NULL ctx");
    if (!u || !v || !items_bias || !users_bias || (nnz > 0 && (!ratings_index || !ratings)) || (n_rows > 0 && !rows))
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_fold_in_funk: NULL array");
    if (side != MFREC_FOLD_USERS && side != MFREC_FOLD_ITEMS)
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_fold_in_funk: side=%d", side);
    if (k <= 0 || ni <= 0 || nu <= 0 || nnz < 0 || n_rows < 0)
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_fold_in_funk: k=%d ni=%d nu=%d nnz=%lld rows=%d",
                               k, ni, nu, (long long)nnz, n_rows);
    const bool by_user = side == MFREC_FOLD_USERS;
    const int tc = by_user ? 0 : 1;   // column of ratings_index naming the trained row; 1 - tc the frozen one
    FoldSelection sel;
    MF_TRY(sel.count(ctx, "mfrec_fold_in_funk", side, ratings_index, nnz, ni, nu, rows, n_rows));
    const std::vector<int64_t> &rptr = sel.rptr;
    for (int32_t p = 0; p < n_rows; ++p)
        if (rptr[p + 1] == rptr[p])   // mfrec_train_funk refuses nnz = 0 too
            return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG,
                                   "mfrec_fold_in_funk: row %d (rows[%d]) has no ratings (the reference loops forever on 0/0)",
                                   rows[p], p);
    MF_CUDA(ctx, cudaSetDevice(ctx->device));
    if (n_rows == 0) return MFREC_OK;
    const int64_t nsel = sel.nsel();
    sel.gather(ratings_index, ratings, nnz);
    // the listed rows and the frozen rows their ratings name, row-major (a lane reads whole rows)
    FoldRows g;
    g.gather(k, true, u, v, items_bias, users_bias, ni, nu, sel.idx.data(), nsel);
    std::vector<double> &tf = by_user ? g.v : g.u;
    const std::vector<double> &tb = by_user ? g.ub : g.ib, &ff = by_user ? g.u : g.v, &fbv = by_user ? g.ib : g.ub;

    // jobs: the longest rows first (list order among equal counts), 32 to a block; a block's
    // per-rating arrays are 32 x (its first job's count) long, lane-interleaved
    std::vector<int32_t> order(n_rows);
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](int32_t a, int32_t b) {
        return rptr[a + 1] - rptr[a] > rptr[b + 1] - rptr[b];
    });
    const int32_t n_blocks = (n_rows + 31) / 32;
    std::vector<int64_t> warp_off((size_t)n_blocks + 1, 0);
    for (int32_t w = 0; w < n_blocks; ++w) {
        const int32_t p = order[(size_t)w * 32];
        warp_off[w + 1] = warp_off[w] + 32 * (rptr[p + 1] - rptr[p]);
    }
    const int64_t slots = warp_off[n_blocks];
    std::vector<int32_t> job_row(n_rows), job_cnt(n_rows), fidx(slots, 0);
    std::vector<double> rv(slots, 0.0);
    for (int32_t j = 0; j < n_rows; ++j) {
        const int32_t p = order[j];
        const int64_t a = rptr[p], q0 = warp_off[j / 32] + (j % 32);
        job_row[j] = g.idx[2 * a + tc];
        job_cnt[j] = (int32_t)(rptr[p + 1] - a);
        for (int64_t n = 0; n < job_cnt[j]; ++n) {
            fidx[q0 + 32 * n] = g.idx[2 * (a + n) + 1 - tc];
            rv[q0 + 32 * n] = sel.r[a + n];
        }
    }

    cudaStream_t st = ctx->stream;
    DevBuf<double> d_tf, d_tb, d_ff, d_fb, d_rv, d_base, d_so, d_ss, d_fr;
    DevBuf<int32_t> d_row, d_cnt, d_fidx, d_fe;
    DevBuf<int64_t> d_off;
    MF_CUDA(ctx, d_tf.alloc(tf.size(), st));
    MF_CUDA(ctx, d_tb.alloc(tb.size(), st));
    MF_CUDA(ctx, d_ff.alloc(ff.size(), st));
    MF_CUDA(ctx, d_fb.alloc(fbv.size(), st));
    MF_CUDA(ctx, d_rv.alloc(slots, st));
    MF_CUDA(ctx, d_base.alloc(slots, st));
    MF_CUDA(ctx, d_so.alloc(slots, st));
    MF_CUDA(ctx, d_ss.alloc(slots, st));
    MF_CUDA(ctx, d_fidx.alloc(slots, st));
    MF_CUDA(ctx, d_row.alloc(n_rows, st));
    MF_CUDA(ctx, d_cnt.alloc(n_rows, st));
    MF_CUDA(ctx, d_off.alloc((size_t)n_blocks + 1, st));
    MF_CUDA(ctx, d_fe.alloc((size_t)n_rows * k, st));
    MF_CUDA(ctx, d_fr.alloc((size_t)n_rows * k, st));
    MF_CUDA(ctx, cudaMemcpyAsync(d_tf.p, tf.data(), tf.size() * 8, cudaMemcpyHostToDevice, st));
    MF_CUDA(ctx, cudaMemcpyAsync(d_tb.p, tb.data(), tb.size() * 8, cudaMemcpyHostToDevice, st));
    MF_CUDA(ctx, cudaMemcpyAsync(d_ff.p, ff.data(), ff.size() * 8, cudaMemcpyHostToDevice, st));
    MF_CUDA(ctx, cudaMemcpyAsync(d_fb.p, fbv.data(), fbv.size() * 8, cudaMemcpyHostToDevice, st));
    MF_CUDA(ctx, cudaMemcpyAsync(d_rv.p, rv.data(), (size_t)slots * 8, cudaMemcpyHostToDevice, st));
    MF_CUDA(ctx, cudaMemcpyAsync(d_fidx.p, fidx.data(), (size_t)slots * 4, cudaMemcpyHostToDevice, st));
    MF_CUDA(ctx, cudaMemcpyAsync(d_row.p, job_row.data(), (size_t)n_rows * 4, cudaMemcpyHostToDevice, st));
    MF_CUDA(ctx, cudaMemcpyAsync(d_cnt.p, job_cnt.data(), (size_t)n_rows * 4, cudaMemcpyHostToDevice, st));
    MF_CUDA(ctx, cudaMemcpyAsync(d_off.p, warp_off.data(), ((size_t)n_blocks + 1) * 8, cudaMemcpyHostToDevice, st));
    auto launch = by_user ? funk_fold_in_kernel<MFREC_FOLD_USERS> : funk_fold_in_kernel<MFREC_FOLD_ITEMS>;
    launch<<<n_blocks, 32, 0, st>>>(min_epochs, min_improvement, k, f_init, learning_rate, K, overall_avg,
                                    d_tf.p, d_tb.p, d_ff.p, d_fb.p, d_row.p, d_cnt.p, d_off.p, d_fidx.p, d_rv.p,
                                    d_base.p, d_so.p, d_ss.p, n_rows, d_fe.p, d_fr.p);
    MF_LAUNCH_CHECK(ctx);
    std::vector<int32_t> h_fe((size_t)n_rows * k);
    std::vector<double> h_fr((size_t)n_rows * k);
    MF_CUDA(ctx, cudaMemcpyAsync(tf.data(), d_tf.p, tf.size() * 8, cudaMemcpyDeviceToHost, st));
    MF_CUDA(ctx, cudaMemcpyAsync(h_fe.data(), d_fe.p, h_fe.size() * 4, cudaMemcpyDeviceToHost, st));
    MF_CUDA(ctx, cudaMemcpyAsync(h_fr.data(), d_fr.p, h_fr.size() * 8, cudaMemcpyDeviceToHost, st));
    MF_CUDA(ctx, cudaStreamSynchronize(st));
    // only the listed rows go back: the frozen side, both bias arrays and every unlisted row are
    // never written
    if (by_user) g.scatter(nullptr, v, nullptr, nullptr, ni, nu);
    else g.scatter(u, nullptr, nullptr, nullptr, ni, nu);
    for (int32_t j = 0; j < n_rows; ++j) {
        const size_t p = order[j];
        if (feature_epochs) std::copy(h_fe.begin() + (size_t)j * k, h_fe.begin() + (size_t)(j + 1) * k, feature_epochs + p * k);
        if (feature_rmse) std::copy(h_fr.begin() + (size_t)j * k, h_fr.begin() + (size_t)(j + 1) * k, feature_rmse + p * k);
    }
    return MFREC_OK;
}
