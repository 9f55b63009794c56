// Ratings layout: COO -> block-bucketed, user-sorted COO resident in HBM.
//
// GPU counterpart of BaseRecommender.get_ratings (reference base.py:1115-1131): instead of one
// shuffled list walked by one thread, ratings are bucketed so that the SGD kernel can run
// B * W warps that never touch the same user row or item row at the same time (the DSGD /
// cuMF_SGD block schedule), see sgd.cu.
//
//   users  -> B row blocks      x W row groups      (balanced by degree, LPT)
//   items  -> G slabs x B column blocks x W column groups
//   bucket(slab g, row block rb, column block cb, phase p, worker w) holds the ratings of
//   row group (rb, w) x column group (cb, (w + p) mod W), sorted by (user, item) so that
//   ratings of one user are adjacent (sgd.cu keeps that user's row in registers).  (A bucket is
//   one warp's serial work, so any order inside it is legal; see the key layout below for the
//   order that was measured against this one.)
//   Buckets are stored in (g, rb, cb, w, p) order -- worker-major, so the W buckets one warp
//   walks through are one contiguous stream -- each starting on a 16-byte boundary so the
//   warp can pull the stream through shared memory with cp.async.bulk.
//
// Users and items are relabelled ("packed ids") so each group is a contiguous id range; the
// factor matrices live in HBM in packed-id order, which makes every column block's Q tile one
// contiguous chunk.
//
// Steps (all HBM-bound integer work):
//   1. degree histograms + index validation                 (1 pass over idx)
//   2. host: hierarchical LPT partition of users / items     (O(n log B), n = nu + ni)
//   3. 64-bit key = bucket | packed user | packed item       (1 pass)
//   4. stable LSD radix sort of (key, input position)        (cub::DeviceRadixSort)
//   5. bucket histogram -> padded offsets                    (1 pass + scan)
//   6. gather ratings into the packed array                  (1 pass)
#include <algorithm>
#include <cstring>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <numeric>
#include <queue>

#include "common.cuh"
#include "partition.h"

namespace {

__global__ void degree_kernel(const int32_t *__restrict__ idx, int64_t nnz, int32_t ni, int32_t nu,
                              int32_t *__restrict__ deg_u, int32_t *__restrict__ deg_i,
                              int32_t *__restrict__ bad)
{
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; n < nnz; n += stride) {
        const int2 ui = reinterpret_cast<const int2 *>(idx)[n];
        if (ui.x < 0 || ui.x >= nu || ui.y < 0 || ui.y >= ni) {
            atomicOr(bad, 1);
            continue;
        }
        atomicAdd(&deg_u[ui.x], 1);
        atomicAdd(&deg_i[ui.y], 1);
    }
}

struct KeyLayout {
    int bits_i, bits_u, bits_b;
    int W, B;
};

// which copy of a split item a user's rating trains (any fixed function of the user will do: the
// copies only have to see disjoint, similarly sized shares of the item's ratings)
__host__ __device__ inline uint32_t copy_of_user(uint32_t user, uint32_t copies)
{
    uint32_t x = user * 0x9e3779b1u;
    x ^= x >> 15;
    x *= 0x85ebca77u;
    x ^= x >> 13;
    return x % copies;
}

__global__ void key_kernel(const int32_t *__restrict__ idx, int64_t nnz,
                           const int32_t *__restrict__ user_perm,
                           const int32_t *__restrict__ item_perm,   // [ni_v] virtual item -> packed id
                           const int32_t *__restrict__ user_group,  // packed row group  [nu]
                           const int32_t *__restrict__ item_group,  // packed col group  [ni_v]
                           const int32_t *__restrict__ item_vbase,  // [ni + 1] first virtual id of each item
                           KeyLayout kl, uint64_t *__restrict__ keys, uint32_t *__restrict__ vals)
{
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; n < nnz; n += stride) {
        int2 ui = reinterpret_cast<const int2 *>(idx)[n];
        {
            const int32_t vb = item_vbase[ui.y], copies = item_vbase[ui.y + 1] - vb;
            ui.y = vb + (copies > 1 ? (int32_t)copy_of_user((uint32_t)ui.x, (uint32_t)copies) : 0);   // virtual item
        }
        const int rg = user_group[ui.x], cg = item_group[ui.y];
        const int rb = rg / kl.W, wr = rg % kl.W;
        const int cbg = cg / kl.W, wc = cg % kl.W;   // cbg = slab * B + local column block
        const int slab = cbg / kl.B, cbl = cbg % kl.B;
        const int p = (wc - wr + kl.W) % kl.W;
        const uint64_t bucket =
            ((((uint64_t)slab * kl.B + rb) * kl.B + cbl) * kl.W + wr) * kl.W + p;
        const uint64_t pu = (uint32_t)user_perm[ui.x], pi = (uint32_t)item_perm[ui.y];
        keys[n] = (bucket << (kl.bits_u + kl.bits_i)) | (pu << kl.bits_i) | pi;   // bucket, then user, then item
        vals[n] = (uint32_t)n;
    }
}

__global__ void bucket_hist_kernel(const uint64_t *__restrict__ keys, int64_t nnz, int shift,
                                   int32_t *__restrict__ cnt)
{
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; n < nnz; n += stride)
        atomicAdd(&cnt[keys[n] >> shift], 1);
}

__global__ void pad_counts_kernel(const int32_t *__restrict__ cnt, int64_t nb,
                                  int64_t *__restrict__ raw, int64_t *__restrict__ padded,
                                  int32_t *__restrict__ widest)
{
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int32_t c = 0;
    if (b < nb) {
        c = cnt[b];
        raw[b] = c;
        padded[b] = (c + 3) & ~3;
    }
    for (int o = 16; o > 0; o >>= 1) c = max(c, __shfl_xor_sync(0xffffffffu, c, o));
    if ((threadIdx.x & 31) == 0 && c > 0) atomicMax(widest, c);
}

constexpr int32_t kTmpFirst = 1 << 30;   // .u, only between gather_kernel and hint_kernel: first rating of its bucket

template <typename RT>
__global__ void gather_kernel(const uint64_t *__restrict__ keys, const uint32_t *__restrict__ vals,
                              int64_t nnz, const RT *__restrict__ ratings, KeyLayout kl,
                              const int64_t *__restrict__ raw_off,
                              const int64_t *__restrict__ pad_off,
                              PackedRating *__restrict__ packed, int64_t *__restrict__ order)
{
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const uint64_t mask_i = (1ull << kl.bits_i) - 1, mask_u = (1ull << kl.bits_u) - 1;
    for (int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < nnz; s += stride) {
        const uint64_t key = keys[s];
        const uint32_t src = vals[s];
        const uint64_t b = key >> (kl.bits_u + kl.bits_i);
        const int64_t at = s - raw_off[b];
        const int64_t dst = pad_off[b] + at;
        PackedRating pr;
        pr.u = (int32_t)((key >> kl.bits_i) & mask_u) | (at == 0 ? kTmpFirst : 0);
        pr.i = (int32_t)(key & mask_i);
        pr.r = (float)ratings[src];
        packed[dst] = pr;
        if (order) order[dst] = (int64_t)src;
    }
}

// Hints for the SGD kernel (common.cuh), from the FINAL order of the packed array.  The prefetch
// window of a warp reaches back at most 32 stream positions; the entries before a position in
// memory are its predecessors in its warp's stream, or -- at the head of a stream -- the tail of
// another worker's stream, whose users (another row group) never match.
__global__ void hint_kernel(PackedRating *__restrict__ packed, int64_t n)
{
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += stride) {
        const int32_t u_raw = packed[j].u, i_raw = packed[j].i;
        if (i_raw & kFlagPad) continue;
        const int32_t u = u_raw & kIdMask, it = i_raw & kIdMask;
        const bool first = (u_raw & kTmpFirst) != 0;
        bool adjacent = false, same_item = false, stale = false;
        if (!first) {   // (a bucket's ratings are contiguous: j - 1 is its previous rating)
            adjacent = (packed[j - 1].u & kIdMask) == u;
            same_item = (packed[j - 1].i & kIdMask) == it;
        }
        const int64_t lo = j >= 32 ? j - 32 : 0;
        for (int64_t q = j - 1; q >= lo && !stale; --q) {
            if (adjacent && q == j - 1) continue;
            const int32_t qi = packed[q].i;
            if (qi & kFlagPad) continue;
            stale = (packed[q].u & kIdMask) == u;
        }
        if (adjacent && stale) {
            // the user occurs both right before and further back: the registers hold the latest row
            stale = false;
        }
        int32_t flags = 0;
        if (adjacent) flags |= kFlagAdjUser;
        if (stale) flags |= kFlagStale;
        if (same_item) flags |= kFlagSameItem;
        packed[j].i = i_raw | flags;
        if (first) packed[j].u = u;   // the temporary marker must not reach the kernel (readers above mask it off)
    }
}

// max |rating| over the packed array (non-negative floats order like their bit patterns)
__global__ void max_abs_rating_kernel(const PackedRating *__restrict__ packed, int64_t n,
                                      int32_t *__restrict__ out_bits)
{
    int32_t mx = 0;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += stride)
        mx = max(mx, __float_as_int(fabsf(packed[j].r)));
    for (int o = 16; o > 0; o >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((threadIdx.x & 31) == 0) atomicMax(out_bits, mx);
}

// every slot starts as padding; gather_kernel overwrites the real ratings
__global__ void fill_padding_kernel(PackedRating *__restrict__ packed, int64_t n)
{
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    PackedRating pad;
    pad.u = 0; pad.i = kFlagPad; pad.r = 0.f;
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += stride) packed[j] = pad;
}

// classify every aligned quad (buckets are quad aligned, so a quad never spans two buckets)
__global__ void quad_type_kernel(PackedRating *__restrict__ packed, int64_t n_quads,
                                 unsigned long long *__restrict__ type_count)
{
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    int mine[4] = {0, 0, 0, 0};
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < n_quads; q += stride) {
        const int4 *src = reinterpret_cast<const int4 *>(packed + q * 4);
        const int4 a = src[0], b = src[1], c = src[2];
        const int i0 = a.y, i1 = b.x, i2 = b.w, i3 = c.z;
        const int any = i0 | i1 | i2 | i3;
        int type = kQuadGeneric;
        if (!(any & (kFlagPad | kFlagStale))) {
            const int m0 = i0 & kIdMask;
            const bool one_item = (i1 & kIdMask) == m0 && (i2 & kIdMask) == m0 && (i3 & kIdMask) == m0;
            type = (one_item && !(any & kFlagAdjUser)) ? kQuadChain : kQuadClean;
            const int m1 = i1 & kIdMask, m2 = i2 & kIdMask, m3 = i3 & kIdMask;
            if (!(any & kFlagAdjUser) && m0 != m1 && m0 != m2 && m0 != m3 && m1 != m2 && m1 != m3 && m2 != m3)
                type = kQuadIndep;
        }
        packed[q * 4].u = (a.x & kIdMask) | (type << kQuadShift);
        if (!(i0 & kFlagPad)) mine[type] += 1;   // statistics (empty quads excluded)
    }
#pragma unroll
    for (int t = 0; t < 4; ++t) {
        const int tot = __reduce_add_sync(0xffffffffu, mine[t]);
        if ((threadIdx.x & 31) == 0 && tot) atomicAdd(type_count + t, (unsigned long long)tot);
    }
}

__global__ void fill_i64_kernel(int64_t *p, int64_t n, int64_t v)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

int bits_for(int64_t n)
{
    int b = 1;
    while ((1ll << b) < n) ++b;
    return b;
}

// sort key of an id: heaviest first, ties in a seeded pseudo-random order
__global__ void degree_key_kernel(const int32_t *__restrict__ deg, int32_t n, uint64_t seed,
                                  uint64_t *__restrict__ keys, int32_t *__restrict__ ids)
{
    const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint64_t x = seed ^ (uint64_t)i;
    x += 0x9e3779b97f4a7c15ull;
    x = (x ^ (x >> 30)) * 0xbf58476d1ce4e5b9ull;
    x = (x ^ (x >> 27)) * 0x94d049bb133111ebull;
    x ^= x >> 31;
    keys[i] = ((uint64_t)(0xffffffffu - (uint32_t)deg[i]) << 32) | (x >> 32);
    ids[i] = i;
}

struct PackHost {
    std::vector<int32_t> deg_u, deg_i, deg_v, ug, up, ig, ip, sorted_u, sorted_i;
    mfrec_part::Workspace ws_u, ws_i;
    // pinned staging for the partition tables: the device PULLS them with a kernel instead of a
    // host -> device copy, which would queue on the copy engine behind the caller's rating values
    // (hundreds of MB in flight on the copy stream) and stall the sort for up to their duration
    int32_t *pinned = nullptr;
    size_t pinned_cap = 0;
    ~PackHost() { if (pinned) cudaFreeHost(pinned); }
    cudaError_t reserve(size_t n)
    {
        if (n <= pinned_cap) return cudaSuccess;
        if (pinned) cudaFreeHost(pinned);
        pinned = nullptr;
        pinned_cap = 0;
        cudaError_t e = cudaHostAlloc((void **)&pinned, n * 4, cudaHostAllocDefault);
        if (e == cudaSuccess) pinned_cap = n;
        return e;
    }
};

// copies n 32-bit words from pinned (mapped) host memory: SM loads over PCIe, no copy engine
__global__ void pull_host_kernel(const int32_t *__restrict__ src, int32_t *__restrict__ dst, int64_t n)
{
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += stride) dst[j] = src[j];
}

// ids sorted heaviest first -> host vector.  deg_dev may be overridden by deg_host (multi-GPU:
// global item degrees), in which case it is uploaded first.
int sorted_by_degree(mfrec_ctx *ctx, const int32_t *deg_dev, int32_t n, uint64_t seed,
                     std::vector<int32_t> &sorted)
{
    cudaStream_t st = ctx->stream;
    DevBuf<uint64_t> ka, kb;
    DevBuf<int32_t> va, vb;
    MF_CUDA(ctx, ka.alloc(n, st));
    MF_CUDA(ctx, kb.alloc(n, st));
    MF_CUDA(ctx, va.alloc(n, st));
    MF_CUDA(ctx, vb.alloc(n, st));
    degree_key_kernel<<<(n + 255) / 256, 256, 0, st>>>(deg_dev, n, seed, ka.p, va.p);
    MF_LAUNCH_CHECK(ctx);
    cub::DoubleBuffer<uint64_t> dk(ka.p, kb.p);
    cub::DoubleBuffer<int32_t> dv(va.p, vb.p);
    size_t tmp_bytes = 0;
    MF_CUDA(ctx, cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, dk, dv, n, 0, 64, st));
    DevBuf<char> tmp;
    MF_CUDA(ctx, tmp.alloc(tmp_bytes, st));
    MF_CUDA(ctx, cub::DeviceRadixSort::SortPairs(tmp.p, tmp_bytes, dk, dv, n, 0, 64, st));
    ctx->launches += 10;
    sorted.resize(n);
    MF_CUDA(ctx, cudaMemcpyAsync(sorted.data(), dv.Current(), (size_t)n * 4, cudaMemcpyDeviceToHost, st));
    MF_CUDA(ctx, cudaStreamSynchronize(st));
    return MFREC_OK;
}

}  // namespace

extern "C" void mfrec_ratings_destroy(mfrec_ratings *r)
{
    if (!r) return;
    cudaSetDevice(r->device);
    cudaStream_t st = r->ctx->stream;
    void *ptrs[] = {r->user_perm, r->item_perm, r->col_start, r->packed, r->bucket_off, r->bucket_cnt, r->order,
                    r->item_vbase, r->item_rows, r->vitem_src, r->hot_off, r->hot_rows};
    for (void *q : ptrs)
        if (q) cudaFreeAsync(q, st);
    mfrec_ctx_release(r->ctx);
    delete r;
}

extern "C" int mfrec_ratings_pack(mfrec_ctx *ctx, const int32_t *ratings_index, const void *ratings,
                                  int ratings_are_f32, int is_device, int64_t nnz, int32_t ni,
                                  int32_t nu, const int64_t *item_degree, const mfrec_opts *opts,
                                  mfrec_ratings **out)
{
    if (!ctx || !out) return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_ratings_pack: NULL argument");
    *out = nullptr;
    if (nnz < 0 || ni <= 0 || nu <= 0 || (nnz > 0 && (!ratings_index || !ratings)))
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_ratings_pack: nnz=%lld ni=%d nu=%d",
                               (long long)nnz, ni, nu);
    if (nnz >= (1ll << 32))
        return mfrec_set_error(ctx, MFREC_ERR_UNSUPPORTED, "mfrec_ratings_pack: nnz >= 2^32 per device");
    if (nu > kIdMask || ni > kIdMask)
        return mfrec_set_error(ctx, MFREC_ERR_UNSUPPORTED, "mfrec_ratings_pack: more than 2^27 users or items");
    MF_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    Tracer tr("pack", st);
    int G = (opts && opts->n_slabs > 0) ? opts->n_slabs : 1;
    // Concurrency P = B * W warps needs P^2 buckets per slab.  Measured on the Netflix shape
    // (DESIGN.md section 5): ~40 ratings per bucket is the sweet spot -- a sub-epoch costs a fixed
    // hand-over (ticket, tile load, write-back) plus the spread of its blocks' work, so with G
    // slabs (G times fewer ratings per sub-epoch) less concurrency wins -- and for a given P it is
    // better to keep one CTA on every SM with fewer warps than full CTAs on some of the SMs.
    int W = (opts && opts->workers > 0) ? opts->workers : 0;
    int B = (opts && opts->row_blocks > 0) ? opts->row_blocks : 0;
    // A DSGD rank (item_degree given) holds one user slice of the matrix, and every rank of the
    // ring must arrive at the SAME B and W (they exchange Q rows by packed position): plan with the
    // average slice, total ratings / G, which every rank computes from the global degrees, not with
    // this rank's own count.  (dsgd.check_layout_agreement verifies the outcome.)
    double nnz_plan = (double)nnz;
    if (item_degree && G > 1) {
        double tot = 0.0;
        for (int32_t i = 0; i < ni; ++i) tot += (double)item_degree[i];
        nnz_plan = tot / G;
    }
    const double want_p = sqrt(nnz_plan / G / 40.0);
    if (W == 0) {
        W = B > 0 ? (int)lround(want_p / B) : (int)lround(want_p / ctx->sm_count);
        W = std::max(4, std::min(W, 10));   // (10 warps: measured best at Netflix shape once hot items are split; 12 is slower)
    }
    if (W > 16) W = 16;  // the SGD kernel is built for at most 16 warps per CTA
    if (B == 0) B = std::max(1, std::min((int)(want_p / W), ctx->sm_count));
    // (a slice with fewer users than B * W only arises in toy cases; ring callers then pass row_blocks)
    B = (int)std::max<int64_t>(1, std::min<int64_t>(B, std::min<int64_t>(nu, ni / G) / W));
    const uint64_t seed = opts ? opts->seed : 0;
    const bool keep_order = opts && opts->keep_order;
    int kpad_hint = (opts && opts->k_hint > 0) ? mfrec_kpad(opts->k_hint) : 256;
    if (kpad_hint < 0) kpad_hint = 256;
    const int storage = opts ? opts->storage : MFREC_STORAGE_F32;
    if (storage < MFREC_STORAGE_F32 || storage > MFREC_STORAGE_BF16)
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_ratings_pack: opts.storage=%d", storage);

    // ---- stage inputs on the device -------------------------------------------------
    DevBuf<int32_t> idx_stage;
    DevBuf<char> r_stage;
    const int32_t *d_idx = ratings_index;
    const void *d_r = ratings;
    const size_t rsz = ratings_are_f32 ? 4 : 8;
    if (!is_device && nnz > 0) {
        MF_CUDA(ctx, idx_stage.alloc((size_t)nnz * 2, ctx->stream));
        MF_CUDA(ctx, r_stage.alloc((size_t)nnz * rsz, ctx->stream));
        MF_TRY(mfrec_copy_h2d(ctx, idx_stage.p, ratings_index, (size_t)nnz * 8, st));
        MF_TRY(mfrec_copy_h2d(ctx, r_stage.p, ratings, (size_t)nnz * rsz, st));
        d_idx = idx_stage.p;
        d_r = r_stage.p;
    }
    const int grid = ctx->sm_count * 8;
    tr.lap("H2D ratings");

    // ---- 1. degrees + validation ------------------------------------------------------
    DevBuf<int32_t> deg_u, deg_i, bad;
    MF_CUDA(ctx, deg_u.alloc(nu, ctx->stream));
    MF_CUDA(ctx, deg_i.alloc(ni, ctx->stream));
    MF_CUDA(ctx, bad.alloc(1, ctx->stream));
    MF_CUDA(ctx, cudaMemsetAsync(deg_u.p, 0, (size_t)nu * 4, st));
    MF_CUDA(ctx, cudaMemsetAsync(deg_i.p, 0, (size_t)ni * 4, st));
    MF_CUDA(ctx, cudaMemsetAsync(bad.p, 0, 4, st));
    if (nnz > 0) {
        degree_kernel<<<grid, 256, 0, st>>>(d_idx, nnz, ni, nu, deg_u.p, deg_i.p, bad.p);
        MF_LAUNCH_CHECK(ctx);
    }
    // host scratch lives in the context: fresh multi-MB vectors would be page-faulted in on every
    // call, which costs more than the partition that fills them
    if (!ctx->pack_host) ctx->pack_host = std::make_shared<PackHost>();
    PackHost &H = *static_cast<PackHost *>(ctx->pack_host.get());
    std::vector<int32_t> &h_deg_u = H.deg_u, &h_deg_i = H.deg_i;
    h_deg_u.resize(nu);
    h_deg_i.resize(ni);
    int32_t h_bad = 0;
    MF_CUDA(ctx, cudaMemcpyAsync(h_deg_u.data(), deg_u.p, (size_t)nu * 4, cudaMemcpyDeviceToHost, st));
    MF_CUDA(ctx, cudaMemcpyAsync(h_deg_i.data(), deg_i.p, (size_t)ni * 4, cudaMemcpyDeviceToHost, st));
    MF_CUDA(ctx, cudaMemcpyAsync(&h_bad, bad.p, 4, cudaMemcpyDeviceToHost, st));
    MF_CUDA(ctx, cudaStreamSynchronize(st));
    if (h_bad)
        return mfrec_set_error(ctx, MFREC_ERR_INDEX,
                               "mfrec_ratings_pack: ratings_index has a user outside [0,%d) or an item outside [0,%d)",
                               nu, ni);
    tr.lap("degrees");
    if (item_degree)
        for (int32_t i = 0; i < ni; ++i)
            h_deg_i[i] = (int32_t)std::min<int64_t>(item_degree[i], INT32_MAX - 1);

    // ---- 2. partition (host) -----------------------------------------------------------
    mfrec_ratings *R = new (std::nothrow) mfrec_ratings();
    if (!R) return mfrec_set_error(ctx, MFREC_ERR_OOM, "mfrec_ratings_pack: host OOM");
    struct Guard {
        mfrec_ratings *r;
        ~Guard() { if (r) mfrec_ratings_destroy(r); }
    } guard{R};
    R->ctx = ctx;
    mfrec_ctx_retain(ctx);
    R->device = ctx->device;
    R->nnz = nnz;
    R->ni = ni;
    R->nu = nu;
    R->G = G;
    R->W = W;
    R->storage = storage;
    std::vector<int32_t> &ug = H.ug, &up = H.up, &ig = H.ig, &ip = H.ip, &sorted_u = H.sorted_u, &sorted_i = H.sorted_i;
    // ---- hot-item copies (DESIGN.md 4.1b) ------------------------------------------------------
    // The ratings of one item are a serial chain (its row changes with every update): the hottest
    // item's ~250k ratings at Netflix shape take as long as everything else together.  An item with
    // more than tau ratings is therefore trained as several COPIES -- virtual items, each fed the
    // ratings of a fixed share of the users -- which the scheduler treats like any other item
    // and which are merged (averaged) after every epoch.  tau = half the weight of an average
    // column group, so no copy dominates its group; a copy keeps at least `split_min_copy` ratings,
    // enough for its row to have converged to the same stationary estimate as its siblings
    // (tools/hot_split_sim.py; tests/test_convergence_gpu.py pins the RMSE against the reference).
    std::vector<int32_t> &h_vbase = R->h_vbase;
    std::vector<int32_t> &h_deg_v = H.deg_v;   // degree of every virtual item: an even share of its item's
    DevBuf<int32_t> deg_v;
    int32_t ni_v = 0;
    MF_TRY(sorted_by_degree(ctx, deg_u.p, nu, seed, sorted_u));
    // copies for the current (G, B, W), their degrees, and the virtual items sorted by degree
    auto plan_copies = [&]() -> int {
        h_vbase.assign((size_t)ni + 1, 0);
        const int split = opts ? opts->split : 0;
        const int64_t min_copy = (opts && opts->split_min_copy > 0) ? opts->split_min_copy : 1024;
        double tot = 0.0;
        for (int32_t i = 0; i < ni; ++i) tot += (double)h_deg_i[i];
        const double tau = std::max(1.0, 0.5 * tot / ((double)G * B * W));   // half a column group's share
        for (int32_t i = 0; i < ni; ++i) {
            int64_t copies = 1;
            if (split != MFREC_SPLIT_OFF && (double)h_deg_i[i] > tau) {
                copies = (int64_t)ceil((double)h_deg_i[i] / tau);
                copies = std::min<int64_t>(copies, std::max<int64_t>(1, h_deg_i[i] / min_copy));
                copies = std::min<int64_t>(copies, 64);
            }
            h_vbase[i + 1] = h_vbase[i] + (int32_t)copies;
        }
        ni_v = h_vbase[ni];
        if (ni_v > kIdMask)
            return mfrec_set_error(ctx, MFREC_ERR_UNSUPPORTED, "mfrec_ratings_pack: more than 2^27 item rows");
        h_deg_v.resize(ni_v);
        for (int32_t i = 0; i < ni; ++i) {
            const int32_t c = h_vbase[i + 1] - h_vbase[i];
            for (int32_t j = 0; j < c; ++j) h_deg_v[h_vbase[i] + j] = h_deg_i[i] / c + (j < h_deg_i[i] % c ? 1 : 0);
        }
        MF_CUDA(ctx, deg_v.alloc(ni_v, ctx->stream));
        // (pulled from pinned memory by a kernel, like the partition tables below: a host -> device copy
        // would queue on the copy engine behind the caller's rating values and stall the sort)
        MF_CUDA(ctx, H.reserve(2 * (size_t)nu + 3 * (size_t)ni_v + 2 * (size_t)ni + 2 + (size_t)G * 148 * 16 + 65536));
        memcpy(H.pinned, h_deg_v.data(), (size_t)ni_v * 4);
        pull_host_kernel<<<std::max<int>(1, std::min<int>(ctx->sm_count * 8, (ni_v + 255) / 256)), 256, 0, st>>>(
            H.pinned, deg_v.p, (int64_t)ni_v);
        MF_LAUNCH_CHECK(ctx);
        return sorted_by_degree(ctx, deg_v.p, ni_v, seed ^ 0x5bd1e995u, sorted_i);
    };
    MF_TRY(plan_copies());
    tr.lap("degree sort");
    // May this call choose the number of slabs?  (A DSGD rank may not: the ring fixes it.)
    const bool free_slabs = !(opts && opts->n_slabs > 0) && !item_degree;
    for (;;) {
        // items on a second host thread while this one does the users (4 threads for their blocks)
        std::thread items([&] {
            mfrec_part::partition_items(h_deg_v, sorted_i, h_deg_i, h_vbase, G, B, W, ig, ip, R->h_col_start, H.ws_i);
        });
        mfrec_part::partition_ids(h_deg_u, sorted_u, B, W, 1, ug, up, R->h_row_start, H.ws_u, 4);
        items.join();
        int32_t widest = 0;
        for (int cb = 0; cb < G * B; ++cb)
            widest = std::max(widest, R->h_col_start[(cb + 1) * W] - R->h_col_start[cb * W]);
        R->max_cb_items = widest;
        // the SGD kernel keeps one column block of Q (kpad floats per row) in shared memory
        const size_t need = mfrec_sgd_smem_bytes(widest, kpad_hint, W, storage == MFREC_STORAGE_F32 ? 4 : 2);
        if (need <= ctx->smem_optin || widest <= 1 || (opts && opts->row_blocks > 0)) break;
        if (free_slabs && B + std::max(1, B / 8) > ctx->sm_count && G < 64) {
            // A catalogue too large for one tile per SM (Yahoo shape: 136k items): cut the items into
            // more LOCAL slabs, processed one after the other inside the same persistent launch, rather
            // than into more column blocks than there are SMs (which would mean one launch per sub-epoch).
            G += 1;
            B = std::min(B, ctx->sm_count);
            MF_TRY(plan_copies());
            continue;
        }
        B += std::max(1, B / 8);   // grow B until the widest block fits
    }
    R->G = G;
    R->ni_v = ni_v;
    tr.lap("host LPT partition");
    R->B = B;
    R->n_buckets = (int64_t)G * B * B * W * W;
    KeyLayout kl;
    kl.bits_i = bits_for(ni_v);
    kl.bits_u = bits_for(nu);
    kl.bits_b = bits_for(R->n_buckets);
    kl.W = W;
    kl.B = B;
    // Order inside a bucket: sorted by (user, item), so a user's ratings are adjacent and its row
    // stays in registers.  Item-sorted ratings dealt round-robin over the quads give more
    // independent quads but were slower, because a user then recurs inside the prefetch window
    // (21.4 vs 15.8 ms per epoch at Netflix shape, profiles/r02h_pack_order_dealt.log).
    if (kl.bits_i + kl.bits_u + kl.bits_b > 64)
        return mfrec_set_error(ctx, MFREC_ERR_UNSUPPORTED,
                               "mfrec_ratings_pack: sort key needs %d bits", kl.bits_i + kl.bits_u + kl.bits_b);

    DevBuf<int32_t> d_ug, d_ig;
    MF_CUDA(ctx, d_ug.alloc(nu, ctx->stream));
    MF_CUDA(ctx, d_ig.alloc(ni_v, ctx->stream));
    // item-side tables: item_perm [ni_v] virtual item -> packed row; item_rows [ni] item -> packed row
    // of its FIRST copy (what readers of the model use: all copies are equal between epochs);
    // vitem_src [ni_v] the item each virtual id is a copy of; hot_off / hot_rows: CSR of the packed
    // rows of every split item (the merge kernel's work list)
    std::vector<int32_t> h_item_rows(ni), h_vsrc(ni_v), h_hot_off(1, 0), h_hot_rows;
    for (int32_t i = 0; i < ni; ++i) {
        h_item_rows[i] = ip[h_vbase[i]];
        for (int32_t v = h_vbase[i]; v < h_vbase[i + 1]; ++v) h_vsrc[v] = i;
        if (h_vbase[i + 1] - h_vbase[i] > 1) {
            for (int32_t v = h_vbase[i]; v < h_vbase[i + 1]; ++v) h_hot_rows.push_back(ip[v]);
            h_hot_off.push_back((int32_t)h_hot_rows.size());
        }
    }
    R->n_hot = (int32_t)h_hot_off.size() - 1;
    MF_CUDA(ctx, cudaMallocAsync((void **)&R->user_perm, ((size_t)nu + 1) * 4, st));
    MF_CUDA(ctx, cudaMallocAsync((void **)&R->item_perm, ((size_t)ni_v + 1) * 4, st));
    MF_CUDA(ctx, cudaMallocAsync((void **)&R->item_rows, ((size_t)ni + 1) * 4, st));
    MF_CUDA(ctx, cudaMallocAsync((void **)&R->item_vbase, ((size_t)ni + 2) * 4, st));
    MF_CUDA(ctx, cudaMallocAsync((void **)&R->vitem_src, ((size_t)ni_v + 1) * 4, st));
    MF_CUDA(ctx, cudaMallocAsync((void **)&R->hot_off, h_hot_off.size() * 4, st));
    MF_CUDA(ctx, cudaMallocAsync((void **)&R->hot_rows, (h_hot_rows.size() + 1) * 4, st));
    MF_CUDA(ctx, cudaMallocAsync((void **)&R->col_start, R->h_col_start.size() * 4, st));
    {
        const size_t ncs = R->h_col_start.size();
        // the previous call's pull kernels have finished: every pack ends with a stream sync
        MF_CUDA(ctx, H.reserve(2 * (size_t)nu + 3 * (size_t)ni_v + 2 * (size_t)ni + 2 + ncs + h_hot_off.size() +
                               h_hot_rows.size()));
        struct Seg { const int32_t *src; int32_t *dst; size_t n; } segs[10] = {
            {ug.data(), d_ug.p, (size_t)nu}, {up.data(), R->user_perm, (size_t)nu},
            {ig.data(), d_ig.p, (size_t)ni_v}, {ip.data(), R->item_perm, (size_t)ni_v},
            {h_item_rows.data(), R->item_rows, (size_t)ni}, {h_vbase.data(), R->item_vbase, (size_t)ni + 1},
            {h_vsrc.data(), R->vitem_src, (size_t)ni_v}, {h_hot_off.data(), R->hot_off, h_hot_off.size()},
            {h_hot_rows.data(), R->hot_rows, h_hot_rows.size()},
            {R->h_col_start.data(), R->col_start, ncs}};
        size_t at = 0;
        for (const Seg &sg : segs) {
            if (sg.n == 0) continue;
            memcpy(H.pinned + at, sg.src, sg.n * 4);
            pull_host_kernel<<<std::max<int>(1, std::min<int>(grid, (int)((sg.n + 255) / 256))), 256, 0, st>>>(
                H.pinned + at, sg.dst, (int64_t)sg.n);
            MF_LAUNCH_CHECK(ctx);
            at += sg.n;
        }
    }

    // ---- 3./4. keys + stable radix sort ------------------------------------------------
    DevBuf<uint64_t> keys_a, keys_b;
    DevBuf<uint32_t> vals_a, vals_b;
    MF_CUDA(ctx, keys_a.alloc(nnz, ctx->stream));
    MF_CUDA(ctx, keys_b.alloc(nnz, ctx->stream));
    MF_CUDA(ctx, vals_a.alloc(nnz, ctx->stream));
    MF_CUDA(ctx, vals_b.alloc(nnz, ctx->stream));
    cub::DoubleBuffer<uint64_t> dkeys(keys_a.p, keys_b.p);
    cub::DoubleBuffer<uint32_t> dvals(vals_a.p, vals_b.p);
    if (nnz > 0) {
        key_kernel<<<grid, 256, 0, st>>>(d_idx, nnz, R->user_perm, R->item_perm, d_ug.p, d_ig.p, R->item_vbase, kl,
                                         keys_a.p, vals_a.p);
        MF_LAUNCH_CHECK(ctx);
        size_t tmp_bytes = 0;
        const int end_bit = kl.bits_i + kl.bits_u + kl.bits_b;
        MF_CUDA(ctx, cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, dkeys, dvals, nnz, 0, end_bit, st));
        DevBuf<char> tmp;
        MF_CUDA(ctx, tmp.alloc(tmp_bytes, ctx->stream));
        MF_CUDA(ctx, cub::DeviceRadixSort::SortPairs(tmp.p, tmp_bytes, dkeys, dvals, nnz, 0, end_bit, st));
        ctx->launches += (end_bit + 7) / 8 * 2 + 1;  // histogram + one onesweep pass per digit
        MF_CUDA(ctx, cudaStreamSynchronize(st));
    }

    tr.lap("keys + radix sort");
    // ---- 5. bucket histogram -> offsets ---------------------------------------------------
    // device-side statistics, read back once at the end: [0..3] quads by type (64-bit), then
    // the bit pattern of the largest |rating| and the widest bucket (32-bit each)
    DevBuf<unsigned long long> d_stats;
    MF_CUDA(ctx, d_stats.alloc(5, ctx->stream));
    MF_CUDA(ctx, cudaMemsetAsync(d_stats.p, 0, 40, st));
    int32_t *d_stats32 = reinterpret_cast<int32_t *>(d_stats.p + 4);
    const int64_t nb = R->n_buckets;
    DevBuf<int64_t> raw_cnt, pad_cnt, raw_off;
    MF_CUDA(ctx, cudaMallocAsync((void **)&R->bucket_cnt, (size_t)nb * 4, st));
    MF_CUDA(ctx, cudaMallocAsync((void **)&R->bucket_off, ((size_t)nb + 1) * 8, st));
    MF_CUDA(ctx, raw_cnt.alloc(nb + 1, ctx->stream));
    MF_CUDA(ctx, pad_cnt.alloc(nb + 1, ctx->stream));
    MF_CUDA(ctx, raw_off.alloc(nb + 1, ctx->stream));
    MF_CUDA(ctx, cudaMemsetAsync(R->bucket_cnt, 0, (size_t)nb * 4, st));
    MF_CUDA(ctx, cudaMemsetAsync(raw_cnt.p, 0, ((size_t)nb + 1) * 8, st));
    MF_CUDA(ctx, cudaMemsetAsync(pad_cnt.p, 0, ((size_t)nb + 1) * 8, st));
    if (nnz > 0) {
        bucket_hist_kernel<<<grid, 256, 0, st>>>(dkeys.Current(), nnz, kl.bits_u + kl.bits_i, R->bucket_cnt);
        MF_LAUNCH_CHECK(ctx);
    }
    pad_counts_kernel<<<(unsigned)ceil_div64(nb, 256), 256, 0, st>>>(R->bucket_cnt, nb, raw_cnt.p, pad_cnt.p,
                                                                      d_stats32 + 1);
    MF_LAUNCH_CHECK(ctx);
    {
        size_t tmp_bytes = 0;
        MF_CUDA(ctx, cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, raw_cnt.p, raw_off.p, nb + 1, st));
        DevBuf<char> tmp;
        MF_CUDA(ctx, tmp.alloc(tmp_bytes, ctx->stream));
        MF_CUDA(ctx, cub::DeviceScan::ExclusiveSum(tmp.p, tmp_bytes, raw_cnt.p, raw_off.p, nb + 1, st));
        MF_CUDA(ctx, cub::DeviceScan::ExclusiveSum(tmp.p, tmp_bytes, pad_cnt.p, R->bucket_off, nb + 1, st));
        ctx->launches += 4;
        MF_CUDA(ctx, cudaStreamSynchronize(st));
    }
    int64_t packed_len = 0;
    MF_CUDA(ctx, cudaMemcpy(&packed_len, R->bucket_off + nb, 8, cudaMemcpyDeviceToHost));
    R->packed_len = packed_len;

    tr.lap("bucket offsets");
    // ---- 6. gather ------------------------------------------------------------------------
    // +16 entries of slack: bulk copies are rounded up to 16 bytes
    MF_CUDA(ctx, cudaMallocAsync((void **)&R->packed, ((size_t)packed_len + 16) * sizeof(PackedRating), st));
    fill_padding_kernel<<<grid, 256, 0, st>>>(R->packed, packed_len + 16);
    MF_LAUNCH_CHECK(ctx);
    if (keep_order) {
        MF_CUDA(ctx, cudaMallocAsync((void **)&R->order, ((size_t)packed_len + 1) * 8, st));
        fill_i64_kernel<<<(unsigned)ceil_div64(packed_len + 1, 256), 256, 0, st>>>(R->order, packed_len, -1);
        MF_LAUNCH_CHECK(ctx);
    }
    if (ctx->values_enqueued.valid()) {   // (pageable values: the background thread has recorded values_ready)
        const int urc = ctx->values_enqueued.get();
        ctx->values_enqueued = {};
        if (urc != MFREC_OK) return urc;
    }
    if (ctx->values_ready) {   // the caller is still copying the rating values on another stream
        cudaEvent_t ev = ctx->values_ready;
        ctx->values_ready = nullptr;
        MF_CUDA(ctx, cudaStreamWaitEvent(st, ev, 0));
    }
    if (nnz > 0) {
        if (ratings_are_f32)
            gather_kernel<float><<<grid, 256, 0, st>>>(dkeys.Current(), dvals.Current(), nnz,
                                                       (const float *)d_r, kl, raw_off.p,
                                                       R->bucket_off, R->packed, R->order);
        else
            gather_kernel<double><<<grid, 256, 0, st>>>(dkeys.Current(), dvals.Current(), nnz,
                                                        (const double *)d_r, kl, raw_off.p,
                                                        R->bucket_off, R->packed, R->order);
        MF_LAUNCH_CHECK(ctx);
    }
    if (packed_len > 0) {
        hint_kernel<<<grid, 256, 0, st>>>(R->packed, packed_len);
        MF_LAUNCH_CHECK(ctx);
        quad_type_kernel<<<grid, 256, 0, st>>>(R->packed, packed_len / 4, d_stats.p);
        MF_LAUNCH_CHECK(ctx);
        // largest |rating| (sizes the fixed-point reduction scale of the SGD kernel)
        max_abs_rating_kernel<<<grid, 256, 0, st>>>(R->packed, packed_len, d_stats32);
        MF_LAUNCH_CHECK(ctx);
    }
    {
        unsigned long long h_stats[5];
        MF_CUDA(ctx, cudaMemcpyAsync(h_stats, d_stats.p, 40, cudaMemcpyDeviceToHost, st));
        MF_CUDA(ctx, cudaStreamSynchronize(st));
        for (int t = 0; t < 4; ++t) R->quad_types[t] = (int64_t)h_stats[t];
        int32_t tail[2];
        memcpy(tail, &h_stats[4], 8);
        memcpy(&R->max_abs_rating, &tail[0], 4);
        R->max_bucket = tail[1];   // widest bucket (diagnostic; bounds the longest serial chain of one phase)
    }
    tr.lap("gather + stats");
    guard.r = nullptr;
    *out = R;
    return MFREC_OK;
}

extern "C" int mfrec_ratings_info(const mfrec_ratings *r, int64_t info[8])
{
    if (!r || !info) return mfrec_set_error(nullptr, MFREC_ERR_BAD_ARG, "mfrec_ratings_info: NULL argument");
    info[0] = r->B;
    info[1] = r->W;
    info[2] = r->G;
    info[3] = r->max_cb_items;
    info[4] = r->nnz;
    info[5] = (int64_t)r->G * r->B;  // kernel launches per epoch
    info[6] = r->max_bucket;
    info[7] = r->packed_len;
    return MFREC_OK;
}

extern "C" int mfrec_ratings_quad_types(const mfrec_ratings *r, int64_t counts[4])
{
    if (!r || !counts) return mfrec_set_error(nullptr, MFREC_ERR_BAD_ARG, "mfrec_ratings_quad_types: NULL argument");
    for (int t = 0; t < 4; ++t) counts[t] = r->quad_types[t];
    return MFREC_OK;
}

extern "C" int mfrec_ratings_perm(mfrec_ctx *ctx, const mfrec_ratings *r, int32_t *user_perm,
                                  int32_t *item_perm)
{
    if (!ctx || !r) return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_ratings_perm: NULL argument");
    MF_CUDA(ctx, cudaSetDevice(ctx->device));
    if (user_perm) MF_CUDA(ctx, cudaMemcpy(user_perm, r->user_perm, (size_t)r->nu * 4, cudaMemcpyDeviceToHost));
    if (item_perm) MF_CUDA(ctx, cudaMemcpy(item_perm, r->item_rows, (size_t)r->ni * 4, cudaMemcpyDeviceToHost));
    return MFREC_OK;
}

extern "C" int mfrec_ratings_order(mfrec_ctx *ctx, const mfrec_ratings *r, int64_t *order)
{
    if (!ctx || !r || !order) return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_ratings_order: NULL argument");
    if (!r->order)
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_ratings_order: pack with opts.keep_order = 1");
    MF_CUDA(ctx, cudaSetDevice(ctx->device));
    MF_CUDA(ctx, cudaMemcpy(order, r->order, (size_t)r->packed_len * 8, cudaMemcpyDeviceToHost));
    return MFREC_OK;
}

extern "C" int mfrec_ratings_offsets(mfrec_ctx *ctx, const mfrec_ratings *r, int64_t *offsets,
                                     int32_t *counts)
{
    if (!ctx || !r) return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_ratings_offsets: NULL argument");
    MF_CUDA(ctx, cudaSetDevice(ctx->device));
    if (offsets)
        MF_CUDA(ctx, cudaMemcpy(offsets, r->bucket_off, ((size_t)r->n_buckets + 1) * 8, cudaMemcpyDeviceToHost));
    if (counts)
        MF_CUDA(ctx, cudaMemcpy(counts, r->bucket_cnt, (size_t)r->n_buckets * 4, cudaMemcpyDeviceToHost));
    return MFREC_OK;
}

extern "C" int mfrec_ratings_packed(mfrec_ctx *ctx, const mfrec_ratings *r, void *out)
{
    if (!ctx || !r || !out) return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_ratings_packed: NULL argument");
    MF_CUDA(ctx, cudaSetDevice(ctx->device));
    MF_CUDA(ctx, cudaMemcpy(out, r->packed, (size_t)r->packed_len * sizeof(PackedRating), cudaMemcpyDeviceToHost));
    // strip the kernel hints: callers see plain ids, padding all-zero
    PackedRating *h = static_cast<PackedRating *>(out);
    for (int64_t j = 0; j < r->packed_len; ++j) {
        h[j].u &= kIdMask;
        h[j].i = (h[j].i & kFlagPad) ? 0 : (h[j].i & kIdMask);
    }
    return MFREC_OK;
}

extern "C" int mfrec_ratings_slab_items(const mfrec_ratings *r, int32_t slab, int32_t *begin, int32_t *end)
{
    if (!r || slab < 0 || slab >= r->G || !begin || !end)
        return mfrec_set_error(nullptr, MFREC_ERR_BAD_ARG, "mfrec_ratings_slab_items: bad argument");
    *begin = r->h_col_start[(size_t)slab * r->B * r->W];
    *end = r->h_col_start[(size_t)(slab + 1) * r->B * r->W];
    return MFREC_OK;
}

extern "C" int mfrec_ratings_copies(const mfrec_ratings *r, int32_t *vbase, int64_t counts[2])
{
    if (!r) return mfrec_set_error(nullptr, MFREC_ERR_BAD_ARG, "mfrec_ratings_copies: NULL argument");
    if (vbase) memcpy(vbase, r->h_vbase.data(), ((size_t)r->ni + 1) * 4);
    if (counts) {
        counts[0] = r->ni_v;
        counts[1] = r->n_hot;
    }
    return MFREC_OK;
}
