// Context, error reporting, resident model and the boundary layout conversion
// ([k][n] float64 host  <->  [n][kpad] float32 device, optionally row-permuted).
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <mutex>
#include <thread>

#include "common.cuh"

static thread_local std::string g_tls_error;

int mfrec_set_error(mfrec_ctx *ctx, int code, const char *fmt, ...)
{
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (ctx) ctx->err = buf;
    g_tls_error = buf;
    return code;
}

double Tracer::now()
{
    timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6;
}
Tracer::Tracer(const char *name, cudaStream_t stream) : st(stream), what(name)
{
    static const bool env = getenv("MFREC_TRACE") != nullptr;   // (initialised once, also when shards start together)
    on = env;
    t0 = last = on ? now() : 0.0;
}
void Tracer::lap(const char *stage)
{
    if (!on) return;
    cudaStreamSynchronize(st);
    const double t = now();
    fprintf(stderr, "[mfrec trace] %s: %-28s %8.2f ms  (t = %8.2f)\n", what, stage, t - last, t - t0);
    last = t;
}

extern "C" int mfrec_abi_version(void) { return MFREC_B200_ABI_VERSION; }

extern "C" const char *mfrec_last_error(const mfrec_ctx *ctx)
{
    return ctx ? ctx->err.c_str() : g_tls_error.c_str();
}

extern "C" int mfrec_ctx_create(int device, mfrec_ctx **out)
{
    if (!out) return mfrec_set_error(nullptr, MFREC_ERR_BAD_ARG, "mfrec_ctx_create: out is NULL");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return mfrec_set_error(nullptr, MFREC_ERR_CUDA,
                               "mfrec_ctx_create: no CUDA device (%s); this library has no CPU path",
                               cudaGetErrorString(e));
    if (device < 0) {
        if (cudaGetDevice(&device) != cudaSuccess) device = 0;
    }
    if (device >= count)
        return mfrec_set_error(nullptr, MFREC_ERR_BAD_ARG, "mfrec_ctx_create: device %d of %d",
                               device, count);
    cudaDeviceProp prop;
    MF_CUDA(nullptr, cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return mfrec_set_error(nullptr, MFREC_ERR_CUDA,
                               "mfrec_ctx_create: device %d is sm_%d%d; kernels are built for sm_100a only",
                               device, prop.major, prop.minor);
    MF_CUDA(nullptr, cudaSetDevice(device));
    mfrec_ctx *ctx = new (std::nothrow) mfrec_ctx();
    if (!ctx) return mfrec_set_error(nullptr, MFREC_ERR_OOM, "mfrec_ctx_create: host OOM");
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    ctx->smem_optin = prop.sharedMemPerBlockOptin;
    ctx->smem_per_sm = prop.sharedMemPerMultiprocessor;
    ctx->coop_launch = prop.cooperativeLaunch;
    {
        // keep freed scratch in the pool between calls: repeated training calls then pay for
        // cudaMalloc / cudaFree only once
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
            uint64_t keep = UINT64_MAX;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
    }
    e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        delete ctx;
        return mfrec_set_error(nullptr, MFREC_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e));
    }
    *out = ctx;
    return MFREC_OK;
}

void mfrec_ctx_retain(mfrec_ctx *ctx) { ctx->refs += 1; }

extern "C" void mfrec_ctx_destroy(mfrec_ctx *ctx)
{
    if (ctx) mfrec_ctx_release(ctx);
}

void mfrec_ctx_release(mfrec_ctx *ctx)
{
    if (--ctx->refs > 0) return;   // a ratings / model object still frees into this stream
    cudaSetDevice(ctx->device);
    if (ctx->stream) {
        cudaStreamSynchronize(ctx->stream);
        cudaStreamDestroy(ctx->stream);
    }
    if (ctx->copy_stream) {
        cudaStreamSynchronize(ctx->copy_stream);
        cudaStreamDestroy(ctx->copy_stream);
    }
    if (ctx->se_scratch) cudaFree(ctx->se_scratch);
    if (ctx->ticks) cudaFree(ctx->ticks);
    delete ctx;
}

extern "C" void *mfrec_ctx_stream(mfrec_ctx *ctx) { return ctx ? (void *)ctx->stream : nullptr; }

extern "C" int mfrec_ctx_sync(mfrec_ctx *ctx)
{
    if (!ctx) return mfrec_set_error(nullptr, MFREC_ERR_BAD_ARG, "mfrec_ctx_sync: NULL ctx");
    MF_CUDA(ctx, cudaSetDevice(ctx->device));
    MF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return MFREC_OK;
}

extern "C" int64_t mfrec_ctx_launch_count(const mfrec_ctx *ctx) { return ctx ? ctx->launches : 0; }

// ---------------------------------------------------------------------------------------
// Layout conversion kernels.  HBM-bound, one pass: reads are coalesced along n (the
// contiguous axis of the reference's feature-major arrays), writes along k (the contiguous
// axis of the device rows), through a padded 32x32 shared tile.
// ---------------------------------------------------------------------------------------
// n_rows rows are written; row j comes from source column src_of[j] (null: j).  Copies of a hot
// item (src_of not injective) sit next to each other, so the reads stay nearly coalesced.
// (T = the rows' storage type: float, or __half / __nv_bfloat16 for 16-bit user-factor rows,
// narrowed with round-to-nearest)
template <typename T> __device__ __forceinline__ T row_narrow(float x);
template <> __device__ __forceinline__ float row_narrow<float>(float x) { return x; }
template <> __device__ __forceinline__ __half row_narrow<__half>(float x) { return __float2half_rn(x); }
template <> __device__ __forceinline__ __nv_bfloat16 row_narrow<__nv_bfloat16>(float x) { return __float2bfloat16_rn(x); }
__device__ __forceinline__ float row_widen(float x) { return x; }
__device__ __forceinline__ float row_widen(__half x) { return __half2float(x); }
__device__ __forceinline__ float row_widen(__nv_bfloat16 x) { return __bfloat162float(x); }

template <typename T>
__global__ void __launch_bounds__(256)
factor_to_rows_kernel(const double *__restrict__ src_kn, int k, int kpad, int32_t n, int32_t n_rows,
                      const int32_t *__restrict__ src_of, const int32_t *__restrict__ perm,
                      T *__restrict__ dst_nk)
{
    __shared__ float tile[32][33];
    const int64_t j0 = (int64_t)blockIdx.x * 32;
    const int f0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
    const int64_t jc = j0 + tx;
    const int64_t col = jc < n_rows ? (src_of ? src_of[jc] : jc) : 0;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int f = f0 + ty + r * 8;
        float val = 0.f;
        if (f < k && jc < n_rows) val = (float)src_kn[(int64_t)f * n + col];
        tile[ty + r * 8][tx] = val;
    }
    __syncthreads();
    n = n_rows;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int64_t j = j0 + ty + r * 8;
        const int f = f0 + tx;
        if (j < n && f < kpad) {
            const int64_t row = perm ? perm[j] : j;
            dst_nk[row * kpad + f] = row_narrow<T>(tile[tx][ty + r * 8]);
        }
    }
}

template <typename T>
__global__ void __launch_bounds__(256)
rows_to_factor_kernel(const T *__restrict__ src_nk, int k, int kpad, int32_t n,
                      const int32_t *__restrict__ perm, double *__restrict__ dst_kn)
{
    __shared__ float tile[32][33];
    const int64_t j0 = (int64_t)blockIdx.x * 32;
    const int f0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int64_t j = j0 + ty + r * 8;
        const int f = f0 + tx;
        float val = 0.f;
        if (j < n && f < kpad) {
            const int64_t row = perm ? perm[j] : j;
            val = row_widen(src_nk[row * kpad + f]);
        }
        tile[ty + r * 8][tx] = val;
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int f = f0 + ty + r * 8;
        const int64_t j = j0 + tx;
        if (f < k && j < n) dst_kn[(int64_t)f * n + j] = (double)tile[tx][ty + r * 8];
    }
}

__global__ void vec_to_dev_kernel(const double *__restrict__ src, int32_t n_rows, const int32_t *__restrict__ src_of,
                                  const int32_t *__restrict__ perm, float *__restrict__ dst)
{
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n_rows) dst[perm ? perm[j] : j] = (float)src[src_of ? src_of[j] : j];
}

__global__ void vec_from_dev_kernel(const float *__restrict__ src, int32_t n,
                                    const int32_t *__restrict__ perm, double *__restrict__ dst)
{
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n) dst[j] = (double)src[perm ? perm[j] : j];
}

// ---- staged copies of large pageable host arrays ----------------------------------------------
namespace {

struct HostStager {
    // T host threads (MFREC_STAGE_THREADS; default: half the host's hardware threads, 2..8), each with
    // NB bounce buffers of CH bytes.  One thread's memcpy moves ~6-10 GB/s of pageable memory; the
    // link takes 55 GB/s.
    static constexpr int TMAX = 16, NB = 2;
    static constexpr size_t CH = (size_t)8 << 20;
    int T = 4;
    char *buf[TMAX][NB] = {};
    cudaEvent_t ev[TMAX][NB] = {};
    bool ready = false;
    std::mutex mu;   // one staged copy at a time per context
    ~HostStager()
    {
        for (int t = 0; t < TMAX; ++t)
            for (int b = 0; b < NB; ++b) {
                if (ev[t][b]) cudaEventDestroy(ev[t][b]);
                if (buf[t][b]) cudaFreeHost(buf[t][b]);
            }
    }
    cudaError_t init()
    {
        if (ready) return cudaSuccess;
        const char *env = getenv("MFREC_STAGE_THREADS");
        const int hw = (int)std::thread::hardware_concurrency();
        T = env ? atoi(env) : std::max(2, std::min(8, hw / 2));
        T = std::max(1, std::min(T, (int)TMAX));
        for (int t = 0; t < T; ++t)
            for (int b = 0; b < NB; ++b) {
                cudaError_t e = cudaHostAlloc((void **)&buf[t][b], CH, cudaHostAllocDefault);
                if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ev[t][b], cudaEventDisableTiming);
                if (e != cudaSuccess) return e;
            }
        ready = true;
        return cudaSuccess;
    }
};

size_t stage_min_bytes()
{
    const char *s = getenv("MFREC_STAGE_MIN_BYTES");   // tests lower it to reach the staged path
    return s ? (size_t)atoll(s) : ((size_t)8 << 20);
}

bool host_is_pageable(const void *p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return true;
    }
    return a.type == cudaMemoryTypeUnregistered;
}

HostStager *stager_of(mfrec_ctx *ctx)
{
    if (!ctx->stager) ctx->stager = std::make_shared<HostStager>();
    return static_cast<HostStager *>(ctx->stager.get());
}

}  // namespace

bool mfrec_host_needs_staging(const void *host, size_t bytes)
{
    return host && bytes >= stage_min_bytes() && host_is_pageable(host);
}

int mfrec_copy_h2d(mfrec_ctx *ctx, void *dst_dev, const void *src_host, size_t bytes, cudaStream_t st)
{
    if (bytes == 0) return MFREC_OK;
    if (bytes < stage_min_bytes() || !host_is_pageable(src_host)) {
        MF_CUDA(ctx, cudaMemcpyAsync(dst_dev, src_host, bytes, cudaMemcpyHostToDevice, st));
        return MFREC_OK;
    }
    HostStager *S = stager_of(ctx);
    std::lock_guard<std::mutex> lock(S->mu);
    MF_CUDA(ctx, S->init());
    const size_t CH = HostStager::CH;
    const size_t nchunks = (bytes + CH - 1) / CH;
    const int device = ctx->device;
    const int T = S->T;
    cudaError_t errs[HostStager::TMAX];
    std::thread workers[HostStager::TMAX];
    for (int t = 0; t < T; ++t) {
        errs[t] = cudaSuccess;
        workers[t] = std::thread([=, &errs]() {
            cudaError_t e = cudaSetDevice(device);
            size_t i = 0;
            for (size_t c = (size_t)t; c < nchunks && e == cudaSuccess; c += (size_t)T, ++i) {
                const int b = (int)(i % HostStager::NB);
                const size_t off = c * CH, n = std::min(CH, bytes - off);
                e = cudaEventSynchronize(S->ev[t][b]);   // the buffer's previous transfer is done
                if (e != cudaSuccess) break;
                memcpy(S->buf[t][b], static_cast<const char *>(src_host) + off, n);
                e = cudaMemcpyAsync(static_cast<char *>(dst_dev) + off, S->buf[t][b], n, cudaMemcpyHostToDevice, st);
                if (e == cudaSuccess) e = cudaEventRecord(S->ev[t][b], st);
            }
            errs[t] = e;
        });
    }
    for (int t = 0; t < T; ++t) workers[t].join();
    for (int t = 0; t < T; ++t) MF_CUDA(ctx, errs[t]);
    return MFREC_OK;
}

int mfrec_copy_d2h(mfrec_ctx *ctx, void *dst_host, const void *src_dev, size_t bytes, cudaStream_t st)
{
    if (bytes == 0) return MFREC_OK;
    if (bytes < stage_min_bytes() || !host_is_pageable(dst_host)) {
        MF_CUDA(ctx, cudaMemcpyAsync(dst_host, src_dev, bytes, cudaMemcpyDeviceToHost, st));
        MF_CUDA(ctx, cudaStreamSynchronize(st));
        return MFREC_OK;
    }
    HostStager *S = stager_of(ctx);
    std::lock_guard<std::mutex> lock(S->mu);
    MF_CUDA(ctx, S->init());
    // what precedes on `st` (the kernels that produce src_dev) is ordered before the copies below
    // because they are enqueued on the same stream
    const size_t CH = HostStager::CH;
    const size_t nchunks = (bytes + CH - 1) / CH;
    const int device = ctx->device;
    const int T = S->T;
    cudaError_t errs[HostStager::TMAX];
    std::thread workers[HostStager::TMAX];
    for (int t = 0; t < T; ++t) {
        errs[t] = cudaSuccess;
        workers[t] = std::thread([=, &errs]() {
            cudaError_t e = cudaSetDevice(device);
            // two chunks in flight per worker: the transfer of chunk i + 1 runs while chunk i is
            // copied out of its bounce buffer
            size_t pend_off[HostStager::NB] = {0, 0}, pend_n[HostStager::NB] = {0, 0};
            bool pend[HostStager::NB] = {false, false};
            size_t i = 0;
            auto drain = [&](int b) {
                if (!pend[b] || e != cudaSuccess) return;
                e = cudaEventSynchronize(S->ev[t][b]);
                if (e == cudaSuccess) memcpy(static_cast<char *>(dst_host) + pend_off[b], S->buf[t][b], pend_n[b]);
                pend[b] = false;
            };
            for (size_t c = (size_t)t; c < nchunks && e == cudaSuccess; c += (size_t)T, ++i) {
                const int b = (int)(i % HostStager::NB);
                drain(b);   // the buffer still holds an earlier chunk: copy it out first
                if (e != cudaSuccess) break;
                const size_t off = c * CH, n = std::min(CH, bytes - off);
                e = cudaMemcpyAsync(S->buf[t][b], static_cast<const char *>(src_dev) + off, n, cudaMemcpyDeviceToHost, st);
                if (e == cudaSuccess) e = cudaEventRecord(S->ev[t][b], st);
                pend_off[b] = off; pend_n[b] = n; pend[b] = e == cudaSuccess;
            }
            for (int b = 0; b < HostStager::NB; ++b) drain(b);
            errs[t] = e;
        });
    }
    for (int t = 0; t < T; ++t) workers[t].join();
    for (int t = 0; t < T; ++t) MF_CUDA(ctx, errs[t]);
    return MFREC_OK;
}

int mfrec_upload_factor(mfrec_ctx *ctx, const double *host_kn, int k, int kpad, int32_t n,
                        const int32_t *perm_dev, float *dst_nk, const double *staged_dev, int32_t n_rows,
                        const int32_t *src_of_dev, int row_kind)
{
    if (n == 0) return MFREC_OK;
    if (n_rows < 0) n_rows = n;
    if (!host_kn) {
        MF_CUDA(ctx, cudaMemsetAsync(dst_nk, 0, (size_t)n_rows * kpad * (row_kind == MFREC_STORAGE_F32 ? 4 : 2), ctx->stream));
        return MFREC_OK;
    }
    DevBuf<double> stage;
    const double *src = staged_dev;
    if (!src) {
        MF_CUDA(ctx, stage.alloc((size_t)k * n, ctx->stream));
        MF_TRY(mfrec_copy_h2d(ctx, stage.p, host_kn, (size_t)k * n * sizeof(double), ctx->stream));
        src = stage.p;
    }
    dim3 grid((unsigned)ceil_div64(n_rows, 32), (unsigned)(kpad / 32));
    if (row_kind == MFREC_STORAGE_F16)
        factor_to_rows_kernel<<<grid, 256, 0, ctx->stream>>>(src, k, kpad, n, n_rows, src_of_dev, perm_dev, reinterpret_cast<__half *>(dst_nk));
    else if (row_kind == MFREC_STORAGE_BF16)
        factor_to_rows_kernel<<<grid, 256, 0, ctx->stream>>>(src, k, kpad, n, n_rows, src_of_dev, perm_dev, reinterpret_cast<__nv_bfloat16 *>(dst_nk));
    else
        factor_to_rows_kernel<<<grid, 256, 0, ctx->stream>>>(src, k, kpad, n, n_rows, src_of_dev, perm_dev, dst_nk);
    MF_LAUNCH_CHECK(ctx);
    if (!staged_dev) MF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));   // the host buffer is borrowed
    return MFREC_OK;
}

int mfrec_download_factor(mfrec_ctx *ctx, const float *src_nk, int k, int kpad, int32_t n,
                          const int32_t *perm_dev, double *host_kn, int row_kind)
{
    if (n == 0 || !host_kn) return MFREC_OK;
    DevBuf<double> stage;
    MF_CUDA(ctx, stage.alloc((size_t)k * n, ctx->stream));
    dim3 grid((unsigned)ceil_div64(n, 32), (unsigned)(kpad / 32));
    if (row_kind == MFREC_STORAGE_F16)
        rows_to_factor_kernel<<<grid, 256, 0, ctx->stream>>>(reinterpret_cast<const __half *>(src_nk), k, kpad, n, perm_dev, stage.p);
    else if (row_kind == MFREC_STORAGE_BF16)
        rows_to_factor_kernel<<<grid, 256, 0, ctx->stream>>>(reinterpret_cast<const __nv_bfloat16 *>(src_nk), k, kpad, n, perm_dev, stage.p);
    else
        rows_to_factor_kernel<<<grid, 256, 0, ctx->stream>>>(src_nk, k, kpad, n, perm_dev, stage.p);
    MF_LAUNCH_CHECK(ctx);
    MF_TRY(mfrec_copy_d2h(ctx, host_kn, stage.p, (size_t)k * n * sizeof(double), ctx->stream));
    return MFREC_OK;
}

int mfrec_upload_vec(mfrec_ctx *ctx, const double *host, int32_t n, const int32_t *perm_dev,
                     float *dst, const double *staged_dev, int32_t n_rows, const int32_t *src_of_dev)
{
    if (n == 0) return MFREC_OK;
    if (n_rows < 0) n_rows = n;
    if (!host) {
        MF_CUDA(ctx, cudaMemsetAsync(dst, 0, (size_t)n_rows * sizeof(float), ctx->stream));
        return MFREC_OK;
    }
    DevBuf<double> stage;
    const double *src = staged_dev;
    if (!src) {
        MF_CUDA(ctx, stage.alloc((size_t)n, ctx->stream));
        MF_CUDA(ctx, cudaMemcpyAsync(stage.p, host, (size_t)n * sizeof(double),
                                     cudaMemcpyHostToDevice, ctx->stream));
        src = stage.p;
    }
    vec_to_dev_kernel<<<(unsigned)ceil_div64(n_rows, 256), 256, 0, ctx->stream>>>(src, n_rows, src_of_dev, perm_dev, dst);
    MF_LAUNCH_CHECK(ctx);
    if (!staged_dev) MF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return MFREC_OK;
}

int mfrec_download_vec(mfrec_ctx *ctx, const float *src, int32_t n, const int32_t *perm_dev,
                       double *host)
{
    if (n == 0 || !host) return MFREC_OK;
    DevBuf<double> stage;
    MF_CUDA(ctx, stage.alloc((size_t)n, ctx->stream));
    vec_from_dev_kernel<<<(unsigned)ceil_div64(n, 256), 256, 0, ctx->stream>>>(src, n, perm_dev, stage.p);
    MF_LAUNCH_CHECK(ctx);
    MF_CUDA(ctx, cudaMemcpyAsync(host, stage.p, (size_t)n * sizeof(double),
                                 cudaMemcpyDeviceToHost, ctx->stream));
    MF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return MFREC_OK;
}

// ---------------------------------------------------------------------------------------
// Resident model
// ---------------------------------------------------------------------------------------
extern "C" void mfrec_model_destroy(mfrec_model *m)
{
    if (!m) return;
    cudaSetDevice(m->device);
    cudaStream_t st = m->ctx->stream;
    void *ptrs[] = {m->Q, m->ib, m->P, m->ub, m->user_perm, m->item_perm, m->hot_off, m->hot_rows};
    for (void *q : ptrs)
        if (q) cudaFreeAsync(q, st);
    mfrec_ctx_release(m->ctx);
    delete m;
}

extern "C" int mfrec_model_create(mfrec_ctx *ctx, const mfrec_ratings *layout, int k, int32_t ni,
                                  int32_t nu, const double *u, const double *v,
                                  const double *items_bias, const double *users_bias,
                                  mfrec_model **out)
{
    if (!ctx || !out) return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_model_create: NULL argument");
    *out = nullptr;
    if (k <= 0 || ni < 0 || nu < 0)
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_model_create: k=%d ni=%d nu=%d", k, ni, nu);
    const int kpad = mfrec_kpad(k);
    if (kpad < 0)
        return mfrec_set_error(ctx, MFREC_ERR_UNSUPPORTED, "mfrec_model_create: k=%d > 256 is not instantiated", k);
    if (layout && (layout->ni != ni || layout->nu != nu))
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG,
                               "mfrec_model_create: layout is %d x %d, model is %d x %d",
                               layout->nu, layout->ni, nu, ni);
    MF_CUDA(ctx, cudaSetDevice(ctx->device));
    mfrec_model *m = new (std::nothrow) mfrec_model();
    if (!m) return mfrec_set_error(ctx, MFREC_ERR_OOM, "mfrec_model_create: host OOM");
    m->ctx = ctx;
    mfrec_ctx_retain(ctx);
    m->device = ctx->device;
    m->k = k;
    m->kpad = kpad;
    m->ni = ni;
    m->nu = nu;
    // with a layout the item side has one row per VIRTUAL item (hot items are trained as several
    // copies, pack.cu); readers address an item through the row of its first copy
    const int32_t ni_rows = layout ? layout->ni_v : ni;
    m->ni_rows = ni_rows;
    m->n_hot = layout ? layout->n_hot : 0;
    m->p_kind = layout ? layout->storage : MFREC_STORAGE_F32;
    const size_t p_elem = m->p_kind == MFREC_STORAGE_F32 ? 4 : 2;
    int rc = MFREC_OK;
    auto fail = [&](int code) {
        mfrec_model_destroy(m);
        return code;
    };
#define MF_M(call)                                                                        \
    do {                                                                                  \
        cudaError_t e__ = (call);                                                         \
        if (e__ != cudaSuccess)                                                           \
            return fail(mfrec_set_error(ctx, e__ == cudaErrorMemoryAllocation ? MFREC_ERR_OOM : MFREC_ERR_CUDA, \
                                        "%s -> %s", #call, cudaGetErrorString(e__)));     \
    } while (0)
    // +64 floats of slack so vector loads of the last row never leave the allocation
    MF_M(cudaMallocAsync((void **)&m->Q, ((size_t)ni_rows * kpad + 64) * sizeof(float), ctx->stream));
    MF_M(cudaMallocAsync((void **)&m->P, ((size_t)nu * kpad + 64) * p_elem, ctx->stream));
    MF_M(cudaMallocAsync((void **)&m->ib, ((size_t)ni_rows + 64) * sizeof(float), ctx->stream));
    MF_M(cudaMallocAsync((void **)&m->ub, ((size_t)nu + 64) * sizeof(float), ctx->stream));
    if (layout) {
        MF_M(cudaMallocAsync((void **)&m->user_perm, ((size_t)nu + 1) * sizeof(int32_t), ctx->stream));
        MF_M(cudaMallocAsync((void **)&m->item_perm, ((size_t)ni + 1) * sizeof(int32_t), ctx->stream));
        MF_M(cudaMemcpyAsync(m->user_perm, layout->user_perm, (size_t)nu * sizeof(int32_t),
                             cudaMemcpyDeviceToDevice, ctx->stream));
        MF_M(cudaMemcpyAsync(m->item_perm, layout->item_rows, (size_t)ni * sizeof(int32_t),
                             cudaMemcpyDeviceToDevice, ctx->stream));
        if (m->n_hot > 0) {
            std::vector<int32_t> off((size_t)m->n_hot + 1);
            MF_M(cudaMemcpyAsync(off.data(), layout->hot_off, off.size() * 4, cudaMemcpyDeviceToHost, ctx->stream));
            MF_M(cudaStreamSynchronize(ctx->stream));
            MF_M(cudaMallocAsync((void **)&m->hot_off, off.size() * 4, ctx->stream));
            MF_M(cudaMallocAsync((void **)&m->hot_rows, ((size_t)off.back() + 1) * 4, ctx->stream));
            MF_M(cudaMemcpyAsync(m->hot_off, layout->hot_off, off.size() * 4, cudaMemcpyDeviceToDevice, ctx->stream));
            MF_M(cudaMemcpyAsync(m->hot_rows, layout->hot_rows, (size_t)off.back() * 4, cudaMemcpyDeviceToDevice, ctx->stream));
        }
    }
#undef MF_M
    // a one-call drop-in may have staged the float64 arrays on the device already (common.cuh)
    const auto staged = ctx->staged;
    ctx->staged = {};
    if (ctx->factors_enqueued.valid()) {   // (pageable arrays: the background thread has recorded staged.ready)
        const int urc = ctx->factors_enqueued.get();
        ctx->factors_enqueued = {};
        if (urc != MFREC_OK) return fail(urc);
    }
    if (staged.ready) {
        cudaError_t we = cudaStreamWaitEvent(ctx->stream, staged.ready, 0);
        if (we != cudaSuccess) return fail(mfrec_set_error(ctx, MFREC_ERR_CUDA, "cudaStreamWaitEvent: %s", cudaGetErrorString(we)));
    }
    // (item rows: every virtual item takes the column of the item it is a copy of)
    if ((rc = mfrec_upload_factor(ctx, u, k, kpad, ni, layout ? layout->item_perm : nullptr, m->Q, staged.u, ni_rows,
                                  layout ? layout->vitem_src : nullptr)) != MFREC_OK) return fail(rc);
    if ((rc = mfrec_upload_factor(ctx, v, k, kpad, nu, m->user_perm, m->P, staged.v, -1, nullptr, m->p_kind)) != MFREC_OK) return fail(rc);
    if ((rc = mfrec_upload_vec(ctx, items_bias, ni, layout ? layout->item_perm : nullptr, m->ib, staged.ib, ni_rows,
                               layout ? layout->vitem_src : nullptr)) != MFREC_OK) return fail(rc);
    if ((rc = mfrec_upload_vec(ctx, users_bias, nu, m->user_perm, m->ub, staged.ub)) != MFREC_OK) return fail(rc);
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess)
        return fail(mfrec_set_error(ctx, MFREC_ERR_CUDA, "model upload: %s", cudaGetErrorString(e)));
    *out = m;
    return MFREC_OK;
}

extern "C" int mfrec_model_read(mfrec_ctx *ctx, const mfrec_model *m, double *u, double *v,
                                double *items_bias, double *users_bias)
{
    if (!ctx || !m) return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_model_read: NULL argument");
    MF_CUDA(ctx, cudaSetDevice(ctx->device));
    MF_TRY(mfrec_download_factor(ctx, m->Q, m->k, m->kpad, m->ni, m->item_perm, u));
    MF_TRY(mfrec_download_factor(ctx, m->P, m->k, m->kpad, m->nu, m->user_perm, v, m->p_kind));
    MF_TRY(mfrec_download_vec(ctx, m->ib, m->ni, m->item_perm, items_bias));
    MF_TRY(mfrec_download_vec(ctx, m->ub, m->nu, m->user_perm, users_bias));
    return MFREC_OK;
}

extern "C" int mfrec_model_device_ptrs(const mfrec_model *m, void *ptrs[4], int64_t dims[3])
{
    if (!m || !ptrs || !dims)
        return mfrec_set_error(nullptr, MFREC_ERR_BAD_ARG, "mfrec_model_device_ptrs: NULL argument");
    ptrs[0] = m->Q;
    ptrs[1] = m->ib;
    ptrs[2] = m->P;
    ptrs[3] = m->ub;
    dims[0] = m->ni_rows;   // rows of Q / ib (item copies included): what a slab exchange addresses
    dims[1] = m->nu;
    dims[2] = m->kpad;
    return MFREC_OK;
}

// ---- serving from several shards (mfrec_model_topn_sweep_multi, mfrec_model_predict_multi) ----------
int mfrec_check_shards(mfrec_ctx *const *ctxs, const mfrec_model *const *models, int n_shards, const char *who)
{
    mfrec_ctx *c0 = ctxs && n_shards >= 1 ? ctxs[0] : nullptr;
    if (!ctxs || !models || n_shards < 1)
        return mfrec_set_error(c0, MFREC_ERR_BAD_ARG, "%s: no shards (n_shards=%d)", who, n_shards);
    if (n_shards > kMaxShards)
        return mfrec_set_error(c0, MFREC_ERR_UNSUPPORTED, "%s: %d shards, at most %d", who, n_shards, kMaxShards);
    for (int s = 0; s < n_shards; ++s) {
        if (!ctxs[s] || !models[s]) return mfrec_set_error(c0, MFREC_ERR_BAD_ARG, "%s: shard %d: NULL context or model", who, s);
        for (int t = 0; t < s; ++t)
            if (ctxs[t] == ctxs[s])
                return mfrec_set_error(c0, MFREC_ERR_BAD_ARG, "%s: shards %d and %d share a context (one in-flight call per context)",
                                       who, t, s);
        const mfrec_model *m = models[s], *m0 = models[0];
        if (m->device != ctxs[s]->device)
            return mfrec_set_error(c0, MFREC_ERR_BAD_ARG, "%s: shard %d: model on device %d, context on device %d", who, s,
                                   m->device, ctxs[s]->device);
        if (m->k != m0->k || m->kpad != m0->kpad || m->ni != m0->ni || m->nu != m0->nu || m->p_kind != m0->p_kind)
            return mfrec_set_error(c0, MFREC_ERR_BAD_ARG, "%s: shard %d: model k=%d ni=%d nu=%d kpad=%d differs from shard 0's "
                                   "k=%d ni=%d nu=%d kpad=%d", who, s, m->k, m->ni, m->nu, m->kpad, m0->k, m0->ni, m0->nu,
                                   m0->kpad);
    }
    return MFREC_OK;
}

int mfrec_run_shards(mfrec_ctx *const *ctxs, int n_shards, const char *who, const std::function<int(int)> &fn)
{
    std::vector<int> rc(n_shards, MFREC_OK);
    std::vector<std::thread> threads;
    std::vector<int> here;   // shards whose thread could not be started run on the calling thread
    threads.reserve(n_shards);
    for (int s = 1; s < n_shards; ++s) {
        try {
            threads.emplace_back([&rc, &fn, s] { rc[s] = fn(s); });
        } catch (const std::system_error &) {
            here.push_back(s);
        }
    }
    rc[0] = fn(0);
    for (int s : here) rc[s] = fn(s);
    for (std::thread &t : threads) t.join();
    for (int s = 0; s < n_shards; ++s)
        if (rc[s] != MFREC_OK) {
            const std::string msg = ctxs[s]->err;
            return mfrec_set_error(ctxs[0], rc[s], "%s: shard %d (device %d): %s", who, s, ctxs[s]->device, msg.c_str());
        }
    return MFREC_OK;
}
