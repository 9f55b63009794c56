// Internal declarations shared by the translation units of libmfrec_b200.so.
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdarg>
#include <cstdio>
#include <future>
#include <memory>
#include <string>
#include <vector>

#include "mfrec_b200.h"

// One packed rating: ids are PACKED (relabelled) user / item ids.
struct __align__(4) PackedRating {
    int32_t u;
    int32_t i;
    float r;
};
static_assert(sizeof(PackedRating) == 12, "rating triple must be 12 bytes");
// Packed ids use the low 27 bits; the packer leaves hints for the SGD kernel in the bits above,
// so that the hot loop needs no run-time hazard detection:
constexpr int32_t kIdMask = 0x07ffffff;
constexpr int32_t kFlagAdjUser = 1 << 27;   // .i : same user as the previous rating of the bucket (its row is
                                            //      in registers)
constexpr int32_t kFlagStale = 1 << 28;     // .i : the user also occurs, NOT adjacently, among the 32 ratings
                                            //      that precede this one in its warp's stream (a prefetched
                                            //      row may be stale)
constexpr int32_t kFlagSameItem = 1 << 29;  // .i : same item as the previous rating of the bucket
constexpr int32_t kFlagPad = 1 << 30;       // .i : alignment padding, not a rating
constexpr int kQuadShift = 28;              // .u of the first entry of an aligned quad, 2 bits:
constexpr int kQuadGeneric = 0;             //      anything (padding, repeated users, ...)
constexpr int kQuadChain = 1;               //      4 ratings of ONE item, 4 distinct fresh users
constexpr int kQuadClean = 2;               //      4 ratings, users fresh or equal to their predecessor, any items
constexpr int kQuadIndep = 3;               //      4 ratings, 4 distinct fresh users, 4 distinct items

struct mfrec_ctx {
    int device = 0;
    int sm_count = 0;
    size_t smem_optin = 0;         // largest dynamic shared memory one CTA may ask for
    size_t smem_per_sm = 0;
    int coop_launch = 0;           // cudaDevAttrCooperativeLaunch
    cudaStream_t stream = nullptr;
    int64_t launches = 0;
    double *se_scratch = nullptr;  // per-CTA squared-error partials of one epoch
    size_t se_cap = 0;
    int32_t *ticks = nullptr;      // per column block hand-over counters of the running SGD launch
    size_t ticks_cap = 0;
    // Overlap of the host -> device copies of a one-call drop-in with the packer (set by the caller,
    // consumed and cleared by the callee): rating values / factor arrays that are being copied on
    // copy_stream into device staging buffers while the context stream already works on the indices.
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t values_ready = nullptr;     // mfrec_ratings_pack waits for it before it reads the values
    struct {
        const double *u = nullptr, *v = nullptr, *ib = nullptr, *ub = nullptr;  // device, [k][n] / [n]
        cudaEvent_t ready = nullptr;
    } staged;                               // mfrec_model_create converts from these instead of copying
    // Host-side gates of the same hand-over when the arrays are PAGEABLE: staging them through the
    // bounce buffers occupies a host thread, so the one-call drop-in does it on a background thread
    // while the calling thread already runs the packer.  An event must have been RECORDED before a
    // stream may wait for it: the consumer first waits (on the host) for the future that the
    // background thread fulfils right after recording the event; its value is an mfrec_status.
    std::shared_future<int> values_enqueued, factors_enqueued;
    int refs = 1;                  // the creator + every live mfrec_ratings / mfrec_model
    std::shared_ptr<void> pack_host;   // host scratch of mfrec_ratings_pack, reused across calls
    std::shared_ptr<void> stager;      // pinned bounce buffers for large pageable host arrays (runtime.cu)
    std::string err;
};
// Objects allocate from the context's stream-ordered pool and free into it, so they keep the
// context alive until the last of them is destroyed.
void mfrec_ctx_retain(mfrec_ctx *ctx);
void mfrec_ctx_release(mfrec_ctx *ctx);

struct mfrec_ratings {
    mfrec_ctx *ctx = nullptr;
    int device = 0;
    int64_t nnz = 0;
    int32_t ni = 0, nu = 0;
    int B = 1, W = 1, G = 1;
    int storage = 0;               // MFREC_STORAGE_* of the user-factor rows of models created with this layout
    int64_t n_buckets = 0;
    int64_t packed_len = 0;        // nnz + alignment padding
    int32_t max_cb_items = 0;      // widest column block (items) -> shared-memory tile size
    int64_t max_bucket = 0;
    float max_abs_rating = 0.f;    // sizes the fixed-point scale of the warp reduction
    int64_t quad_types[4] = {0, 0, 0, 0};  // quads by kQuadGeneric / kQuadChain / kQuadClean / kQuadIndep
    // device
    int32_t ni_v = 0;              // item ROWS = virtual items (hot items are trained as several copies)
    int32_t n_hot = 0;             // items with more than one copy
    int32_t *user_perm = nullptr;  // [nu] old -> packed id
    int32_t *item_perm = nullptr;  // [ni_v] virtual item -> packed row
    int32_t *item_rows = nullptr;  // [ni] item -> packed row of its first copy
    int32_t *item_vbase = nullptr; // [ni + 1] first virtual id of each item
    int32_t *vitem_src = nullptr;  // [ni_v] virtual id -> item
    int32_t *hot_off = nullptr;    // [n_hot + 1] CSR over hot_rows
    int32_t *hot_rows = nullptr;   // packed rows of the copies of every split item
    int32_t *col_start = nullptr;  // [G*B*W + 1] packed item id where each column group begins
    PackedRating *packed = nullptr;
    int64_t *bucket_off = nullptr; // [n_buckets] first packed position (multiple of 4)
    int32_t *bucket_cnt = nullptr; // [n_buckets]
    int64_t *order = nullptr;      // [packed_len] input index (or -1 for padding), optional
    // host mirrors
    std::vector<int32_t> h_row_start;  // [B*W + 1]
    std::vector<int32_t> h_col_start;  // [G*B*W + 1]
    std::vector<int32_t> h_vbase;      // [ni + 1]
};

struct mfrec_model {
    mfrec_ctx *ctx = nullptr;
    int device = 0;
    int k = 0, kpad = 0;
    int32_t ni = 0, nu = 0;
    int p_kind = 0;       // MFREC_STORAGE_*: P is float32 [nu][kpad], or __half / __nv_bfloat16 [nu][kpad]
    int32_t ni_rows = 0;  // rows of Q / ib: ni, or the layout's virtual items (copies of hot items)
    int32_t n_hot = 0;
    int32_t *hot_off = nullptr, *hot_rows = nullptr;   // own copies of the layout's merge list
    float *Q = nullptr;   // [ni_rows][kpad]  item factors
    float *ib = nullptr;  // [ni_rows]
    float *P = nullptr;   // [nu][kpad]  user factors (elements of 4 or 2 bytes, see p_kind)
    float *ub = nullptr;  // [nu]
    int32_t *user_perm = nullptr;  // own copies (nullptr = identity)
    int32_t *item_perm = nullptr;
};

// ---- dependency levels of a window of ratings (sequential schedules, sgd.cu / funk.cu) ------------
// Up to 32 ratings of a stream, one per lane.  Two ratings interact only through the rows / biases of
// a shared user or item, so a rating's level is 1 + the deeper level of the latest EARLIER rating of
// the window with the same user and of the one with the same item (longest path, relaxed until
// nothing changes: as many rounds as there are levels).  Ratings of one level touch disjoint rows
// and may run together; running the levels in order is equivalent to walking the stream.
// Returns this lane's level; lmax = the deepest level of a live lane (0 for an empty window).
#ifdef __CUDACC__
__device__ __forceinline__ int mfrec_window_levels(int user, int item, bool live, int lane, int &lmax)
{
    const unsigned full = 0xffffffffu, below = (1u << lane) - 1u;
    const int pu = 31 - __clz(__match_any_sync(full, live ? user : -1 - lane) & below);   // -1: none
    const int pi = 31 - __clz(__match_any_sync(full, live ? item : -1 - lane) & below);
    int level = 1;
    if (__any_sync(full, pu >= 0 || pi >= 0)) {
        for (;;) {
            const int lu = __shfl_sync(full, level, pu < 0 ? lane : pu);
            const int li = __shfl_sync(full, level, pi < 0 ? lane : pi);
            int nl = 1;
            if (pu >= 0) nl = lu + 1;
            if (pi >= 0) nl = max(nl, li + 1);
            const bool changed = nl != level;
            level = nl;
            if (!__any_sync(full, changed)) break;
        }
    }
    lmax = __reduce_max_sync(full, live ? level : 0);
    return level;
}

// ---- PTX helpers: mbarrier + bulk async copy (TMA, non-tensor form) -------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar)
{
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

// ---- hand-over counters between CTAs of one device (release / acquire at gpu scope) ----------------
__device__ __forceinline__ int ld_acquire_gpu(const int32_t *p)
{
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_gpu(int32_t *p, int v)
{
    asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// ---- score order key of the top-N paths (topn.cu, topn_tc.cu) ---------------------------------------
// monotone map float -> uint32 (larger float -> larger uint) and its inverse
__device__ __forceinline__ uint32_t order_bits(float x)
{
    const uint32_t b = __float_as_uint(x);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float unorder_bits(uint32_t k)
{
    const uint32_t b = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
    return __uint_as_float(b);
}
#endif

// ---- error plumbing -------------------------------------------------------------------
int mfrec_set_error(mfrec_ctx *ctx, int code, const char *fmt, ...);

#define MF_CUDA(ctx, call)                                                                   \
    do {                                                                                     \
        cudaError_t e__ = (call);                                                            \
        if (e__ != cudaSuccess) {                                                            \
            return mfrec_set_error((ctx),                                                    \
                                   e__ == cudaErrorMemoryAllocation ? MFREC_ERR_OOM          \
                                                                    : MFREC_ERR_CUDA,        \
                                   "%s:%d: %s -> %s", __FILE__, __LINE__, #call,             \
                                   cudaGetErrorString(e__));                                 \
        }                                                                                    \
    } while (0)

#define MF_TRY(call)                      \
    do {                                  \
        int rc__ = (call);                \
        if (rc__ != MFREC_OK) return rc__; \
    } while (0)

#define MF_LAUNCH_CHECK(ctx)                 \
    do {                                     \
        (ctx)->launches += 1;                \
        MF_CUDA((ctx), cudaGetLastError());  \
    } while (0)

// Device buffer that frees itself (host-side RAII for scratch allocations).  With a stream the
// memory comes from the device's stream-ordered pool (cudaMallocAsync): no device-wide
// synchronisation on free, and the pool keeps the pages for the next call.
template <typename T>
struct DevBuf {
    T *p = nullptr;
    size_t n = 0;
    cudaStream_t st = nullptr;
    bool pooled = false;
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    ~DevBuf() { release(); }
    cudaError_t alloc(size_t count)
    {
        release();
        n = count;
        pooled = false;
        return cudaMalloc((void **)&p, (count ? count : 1) * sizeof(T));
    }
    cudaError_t alloc(size_t count, cudaStream_t stream)
    {
        release();
        n = count;
        st = stream;
        pooled = true;
        return cudaMallocAsync((void **)&p, (count ? count : 1) * sizeof(T), stream);
    }
    void release()
    {
        if (p) {
            if (pooled) cudaFreeAsync(p, st);
            else cudaFree(p);
        }
        p = nullptr;
        n = 0;
    }
    T *take()
    {
        T *q = p;
        p = nullptr;
        return q;
    }
};

// MFREC_TRACE=1: wall-clock trace of the host-side stages of an entry point, to stderr.
struct Tracer {
    bool on;
    cudaStream_t st;
    const char *what;
    double t0, last;
    static double now();
    Tracer(const char *name, cudaStream_t stream);
    void lap(const char *stage);   // synchronises the stream when tracing, otherwise free
};

static inline int mfrec_kpad(int k)
{
    if (k <= 32) return 32;
    if (k <= 64) return 64;
    if (k <= 128) return 128;
    if (k <= 256) return 256;
    return -1;
}

static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

// sgd.cu
size_t mfrec_sgd_smem_bytes(int tile_rows, int kpad, int W, int p_elem_bytes = 4);

// topn.cu: the exact top-N on a resident model (M may be NULL only when nothing is scored; ni / nu are
// read only then)
int mfrec_topn_on_model(mfrec_ctx *ctx, const mfrec_model *M, int predictor, const int32_t *users, int32_t n_users,
                     int32_t n_candidates, const int64_t *rated_indptr, const int32_t *rated_items, double mu,
                     double min_rating, double max_rating, int32_t N, int32_t *out_items, double *out_scores,
                     int32_t *out_counts, int32_t ni, int32_t nu);

// runtime.cu
// Host <-> device copies of caller-owned arrays.  Page-locked memory goes straight to
// cudaMemcpyAsync; a large PAGEABLE array is staged through pinned bounce buffers by four host
// threads (the runtime's own pageable path is a single-threaded memcpy: ~3x slower).  h2d returns
// when every chunk is enqueued on `st` (the host array may then be reused), d2h when the data
// is in `dst_host`.
int mfrec_copy_h2d(mfrec_ctx *ctx, void *dst_dev, const void *src_host, size_t bytes, cudaStream_t st);
int mfrec_copy_d2h(mfrec_ctx *ctx, void *dst_host, const void *src_dev, size_t bytes, cudaStream_t st);
// true when mfrec_copy_h2d / mfrec_copy_d2h would stage this array (large and pageable), i.e. block the caller
bool mfrec_host_needs_staging(const void *host, size_t bytes);
// n_rows / src_of_dev: write n_rows rows, row j taken from source column src_of_dev[j] (item copies);
// defaults: one row per source column
int mfrec_upload_factor(mfrec_ctx *ctx, const double *host_kn, int k, int kpad, int32_t n,
                        const int32_t *perm_dev, float *dst_nk, const double *staged_dev = nullptr,
                        int32_t n_rows = -1, const int32_t *src_of_dev = nullptr,
                        int row_kind = MFREC_STORAGE_F32);   // row_kind: element type of dst_nk
int mfrec_download_factor(mfrec_ctx *ctx, const float *src_nk, int k, int kpad, int32_t n,
                          const int32_t *perm_dev, double *host_kn, int row_kind = MFREC_STORAGE_F32);
int mfrec_upload_vec(mfrec_ctx *ctx, const double *host, int32_t n, const int32_t *perm_dev,
                     float *dst, const double *staged_dev = nullptr, int32_t n_rows = -1,
                     const int32_t *src_of_dev = nullptr);
// sgd.cu: average the copies of every split item whose rows lie in [row_lo, row_hi) and write the
// mean back to all of them.  ticks != null: first wait until counters [tick_lo, tick_hi) have reached
// tick_need (a ring rank merges the slab it holds once its neighbour has pushed all of it).
int mfrec_merge_copies(mfrec_ctx *ctx, float *Q, float *ib, int kpad, const int32_t *hot_off,
                       const int32_t *hot_rows, int32_t n_hot, int32_t row_lo, int32_t row_hi,
                       const int32_t *ticks, int32_t tick_lo, int32_t tick_hi, int32_t tick_need,
                       int32_t *abort_flag, unsigned long long wait_ns);
int mfrec_download_vec(mfrec_ctx *ctx, const float *src, int32_t n, const int32_t *perm_dev,
                       double *host);
