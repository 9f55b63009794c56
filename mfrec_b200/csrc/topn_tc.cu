// Top-N sweep on the tensor cores: rows of U.V^T for MANY users x all candidate items
// (BASELINE configs[4]: Netflix-shaped factors, k = 128, all users x all items, top-100).
//
// Same contract as mfrec_topn (topn.cu), which replaces the per-item Python loops of
// MFRecommender.find_recommended_items (mfrec/recommendation/mf.py:144-193) and
// GDRecommender.find_user_top_match (gradient_descent.py:769-802): mask the rated items and the
// item whose id equals the user id, NaN -> 0, drop zeros, score descending, ties by ascending
// item id, first N.  Results are EXACT (fp32 scores as in topn.cu, up to summation order); the tensor cores only
// decide which few hundred items per user are worth scoring exactly:
//
//   1. moments   : mean / covariance of the item rows -> per user a threshold tau_u on
//                  x_ui = p_u.q_i + b_i  such that ~2.2 N items are expected above it, and a bound
//                  eps_u on the bf16 rounding error of x_ui
//   2. pack      : U, V -> bf16 operand tiles, K-major, 128-byte swizzled, laid out in HBM exactly
//                  as the MMA reads them from shared memory (one bulk copy per tile, no tensor map)
//   3. sweep     : tcgen05.mma (kind::f16, bf16 x bf16 -> fp32 in TMEM), 512 users x 64 items per
//                  step; warp-specialised: 1 bulk-copy producer lane, 1 MMA issuer lane, 8
//                  epilogue warps that pull the accumulators with tcgen05.ld and append every
//                  item with x > tau_u to the user's candidate list.  U.V^T is never stored.
//   4. finish    : one CTA per user re-scores its candidates in fp32 with the predictor, applies
//                  the masks, ranks them by counting and CERTIFIES the list: the N-th exact
//                  x must clear tau_u + eps_u, i.e. no item below the threshold can belong to the
//                  top N.  Users that cannot be certified (too few candidates, overflow) are
//                  redone by the exact all-items path of topn.cu.
//
// FLOPs: 2 * users * items * k on the tensor pipe (2.175e15 at Netflix shape); everything else is
// O(users * (k^2 + C * k)) on the CUDA cores.
#include <cuda_bf16.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "common.cuh"

namespace {

constexpr int kBN = 64;          // items per MMA step (UMMA N)
constexpr int kCand = 1024;      // candidate slots per user
constexpr int kEpiWarps = 8;
constexpr int kSweepThreads = 64 + kEpiWarps * 32;   // warp 0 producer, warp 1 MMA, warps 2.. epilogue

// ---- PTX helpers (mbarrier init / expect_tx / wait and bulk copies: common.cuh) ----------------
__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// D[tmem] (+)= A[smem] . B[smem]^T, bf16 inputs, fp32 accumulate; issued by ONE thread
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// mbarrier arrives once every MMA issued so far by this thread has completed
__device__ __forceinline__ void umma_commit(uint64_t *bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// 32 lanes x 32 consecutive fp32 columns of TMEM -> 32 registers per thread (thread = lane)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptor of a K-major, 128-byte-swizzled operand block
// ([rows][64 bf16], 8-row groups 1024 B apart): start >> 4 | LBO = 1 | SBO = 1024 >> 4 |
// version 1 (Blackwell) | layout SWIZZLE_128B (2) in bits [61, 64)
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr)
{
    return (uint64_t)((saddr & 0x3ffffu) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) |
           ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
// Instruction descriptor (kind::f16): D = F32 (bit 4), A = B = BF16 (bits 7, 10), both K-major,
// N >> 3 at bit 17, M >> 4 at bit 24
constexpr uint32_t kIdesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(kBN >> 3) << 17) | ((128u >> 4) << 24);

// ---- 2. operand packing -----------------------------------------------------------------------
// dst = [tile][kb][ROWS][64] bf16 with the 16-byte chunks of every row XOR-swizzled by (row & 7);
// one thread per 16-byte chunk.  Column `bias_col` (if >= 0) takes bias[row] (items) / 1.0 (users).
template <int ROWS>
__global__ void __launch_bounds__(256)
pack_operand_kernel(const float *__restrict__ src, int kpad_src, int k, const int32_t *__restrict__ row_ids,
                    int64_t row0, int64_t n_rows, int64_t n_limit, int KB, int bias_col,
                    const float *__restrict__ bias, __nv_bfloat16 *__restrict__ dst, int64_t n_chunks)
{
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_chunks) return;
    const int c = (int)(g & 7);
    const int64_t rowi = g >> 3;                       // (tile * KB + kb) * ROWS + r
    const int r = (int)(rowi % ROWS);
    const int kb = (int)((rowi / ROWS) % KB);
    const int64_t tile = rowi / ROWS / KB;
    const int64_t local = tile * ROWS + r;
    float vals[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (local < n_rows) {
        const int64_t id = row_ids ? row_ids[row0 + local] : row0 + local;
        if (id < n_limit) {
            const float *s = src + id * kpad_src;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int col = kb * 64 + c * 8 + j;
                if (col < k) vals[j] = s[col];
                else if (col == bias_col) vals[j] = bias ? bias[id] : 1.f;
            }
        }
    }
    uint4 out;
    __nv_bfloat162 h0 = __floats2bfloat162_rn(vals[0], vals[1]), h1 = __floats2bfloat162_rn(vals[2], vals[3]);
    __nv_bfloat162 h2 = __floats2bfloat162_rn(vals[4], vals[5]), h3 = __floats2bfloat162_rn(vals[6], vals[7]);
    out.x = *reinterpret_cast<uint32_t *>(&h0); out.y = *reinterpret_cast<uint32_t *>(&h1);
    out.z = *reinterpret_cast<uint32_t *>(&h2); out.w = *reinterpret_cast<uint32_t *>(&h3);
    reinterpret_cast<uint4 *>(dst)[rowi * 8 + (c ^ (r & 7))] = out;
}

// ---- 1. moments ---------------------------------------------------------------------------------
// item side, augmented row a_i = [q_i, b_i]: sum[f] = sum_i a_if, gram[f][g] = sum_i a_if a_ig over
// the candidate items; fp64 accumulation, one block per (f, g-chunk)
__global__ void __launch_bounds__(256)
item_moments_kernel(const float *__restrict__ Q, const float *__restrict__ ib, int kpad, int ka, int k,
                    int32_t nc, double *__restrict__ sum, double *__restrict__ gram, float *__restrict__ qmax2)
{
    // grid = (ka, ka): block (f, g) reduces over items
    const int f = blockIdx.x, g = blockIdx.y;
    if (g > f) return;
    double acc = 0.0, s = 0.0;
    float m2 = 0.f;
    for (int32_t i = threadIdx.x; i < nc; i += blockDim.x) {
        const float af = f < k ? Q[(size_t)i * kpad + f] : ib[i];
        const float ag = g < k ? Q[(size_t)i * kpad + g] : ib[i];
        acc += (double)af * (double)ag;
        if (g == 0) s += (double)af;
        if (f == 0 && g == 0) {   // this block also finds max |q_i|^2 (+ b_i^2)
            float n2 = 0.f;
            for (int e = 0; e < k; ++e) n2 = fmaf(Q[(size_t)i * kpad + e], Q[(size_t)i * kpad + e], n2);
            if (ka > k) n2 = fmaf(ib[i], ib[i], n2);
            m2 = fmaxf(m2, n2);
        }
    }
    __shared__ double sh[256], sh2[256];
    __shared__ float shm[256];
    sh[threadIdx.x] = acc; sh2[threadIdx.x] = s; shm[threadIdx.x] = m2;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) {
            sh[threadIdx.x] += sh[threadIdx.x + o];
            sh2[threadIdx.x] += sh2[threadIdx.x + o];
            shm[threadIdx.x] = fmaxf(shm[threadIdx.x], shm[threadIdx.x + o]);
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        gram[(size_t)f * ka + g] = sh[0];
        gram[(size_t)g * ka + f] = sh[0];
        if (g == 0) sum[f] = sh2[0];
        if (f == 0 && g == 0) *qmax2 = shm[0];
    }
}

// per user (one warp): mean and variance of x_ui over the candidate items from the item moments,
// tau_u = mean + z * sd, eps_u = 2^-7 * |[p_u, 1]| * max_i |[q_i, b_i]|
__global__ void __launch_bounds__(256)
user_threshold_kernel(const float *__restrict__ P, int kpad, int k, int ka, const int32_t *__restrict__ users,
                      int64_t u0, int32_t n_users, int32_t nu, const double *__restrict__ sum,
                      const double *__restrict__ gram, const float *__restrict__ qmax2, int32_t nc, float z,
                      float *__restrict__ tau, float *__restrict__ eps)
{
    extern __shared__ float cov[];   // [ka][ld] covariance (odd row pitch: no bank conflicts), then [ka] mean
    const int ld = ka | 1;
    float *mean = cov + ka * ld;
    for (int j = threadIdx.x; j < ka * ka; j += blockDim.x) {
        const int f = j / ka, g = j % ka;
        cov[f * ld + g] = (float)(gram[j] / nc - (sum[f] / nc) * (sum[g] / nc));
    }
    for (int j = threadIdx.x; j < ka; j += blockDim.x) mean[j] = (float)(sum[j] / nc);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (w >= n_users) return;
    const int64_t uid = users ? users[u0 + w] : u0 + w;
    if (uid < 0 || uid >= nu) { if (lane == 0) { tau[w] = INFINITY; eps[w] = 0.f; } return; }
    const float *p = P + uid * kpad;
    float m = 0.f, var = 0.f, n2 = 0.f;
    for (int f = lane; f < ka; f += 32) {
        const float pf = f < k ? p[f] : 1.f;
        float row = 0.f;
        for (int g = 0; g < ka; ++g) row = fmaf(cov[f * ld + g], g < k ? p[g] : 1.f, row);
        var = fmaf(pf, row, var);
        m = fmaf(pf, mean[f], m);
        n2 = fmaf(pf, pf, n2);
    }
    for (int o = 16; o > 0; o >>= 1) {
        m += __shfl_xor_sync(0xffffffffu, m, o);
        var += __shfl_xor_sync(0xffffffffu, var, o);
        n2 += __shfl_xor_sync(0xffffffffu, n2, o);
    }
    if (lane == 0) {
        tau[w] = m + z * sqrtf(fmaxf(var, 0.f));
        eps[w] = 0.0078125f * sqrtf(n2) * sqrtf(*qmax2);
    }
}

// The same thresholds where the [ka][ka] covariance does not fit one CTA's shared memory (ka > 240
// with 227 KB per block): the covariance is formed once in global memory, as float values equal to
// user_threshold_kernel's, and read from there through L2.  The covariance is exactly symmetric
// (gram is written symmetrically, the mean product commutes), so a lane reads entry [g][f] for its
// row f: neighbouring lanes read neighbouring floats, in the same order of g as the shared-memory
// kernel, which therefore gives the same tau and eps.
__global__ void __launch_bounds__(256)
item_cov_kernel(const double *__restrict__ sum, const double *__restrict__ gram, int ka, int32_t nc, float *__restrict__ cov)
{
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= ka * ka) return;
    const int f = j / ka, g = j % ka;
    cov[j] = (float)(gram[j] / nc - (sum[f] / nc) * (sum[g] / nc));
}

__global__ void __launch_bounds__(256)
user_threshold_l2_kernel(const float *__restrict__ P, int kpad, int k, int ka, const int32_t *__restrict__ users,
                         int64_t u0, int32_t n_users, int32_t nu, const double *__restrict__ sum,
                         const float *__restrict__ cov, const float *__restrict__ qmax2, int32_t nc, float z,
                         float *__restrict__ tau, float *__restrict__ eps)
{
    const int lane = threadIdx.x & 31;
    const int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (w >= n_users) return;
    const int64_t uid = users ? users[u0 + w] : u0 + w;
    if (uid < 0 || uid >= nu) { if (lane == 0) { tau[w] = INFINITY; eps[w] = 0.f; } return; }
    const float *p = P + uid * kpad;
    float m = 0.f, var = 0.f, n2 = 0.f;
    for (int f = lane; f < ka; f += 32) {
        const float pf = f < k ? p[f] : 1.f;
        float row = 0.f;
        for (int g = 0; g < ka; ++g) row = fmaf(cov[g * ka + f], g < k ? p[g] : 1.f, row);
        var = fmaf(pf, row, var);
        m = fmaf(pf, (float)(sum[f] / nc), m);
        n2 = fmaf(pf, pf, n2);
    }
    for (int o = 16; o > 0; o >>= 1) {
        m += __shfl_xor_sync(0xffffffffu, m, o);
        var += __shfl_xor_sync(0xffffffffu, var, o);
        n2 += __shfl_xor_sync(0xffffffffu, n2, o);
    }
    if (lane == 0) {
        tau[w] = m + z * sqrtf(fmaxf(var, 0.f));
        eps[w] = 0.0078125f * sqrtf(n2) * sqrtf(*qmax2);
    }
}

// ---- 3. the sweep -------------------------------------------------------------------------------
struct SweepParams {
    const __nv_bfloat16 *A;     // [groups * NA][KB][128][64]   user tiles of this batch
    const __nv_bfloat16 *B;     // [n_btiles][KB][64][64]       item tiles
    const float *tau;           // [n_users]
    int32_t *cand;              // [n_users][kCand]  item ids above the threshold, ascending
    int32_t *cand_cnt;          // [n_users]  (kCand + 1 = overflow: the list is incomplete)
    int32_t n_users, n_groups, n_btiles, nc;
};

template <int KB, int NA, int kBStages>   // K blocks of 64, user tiles per CTA, B tiles in flight
__global__ void __launch_bounds__(kSweepThreads, 1)
topn_sweep_kernel(const SweepParams p)
{
    constexpr uint32_t A_TILE = KB * 128 * 128;      // bytes: KB blocks of 128 rows x 128 B
    constexpr uint32_t B_TILE = KB * kBN * 128;
    constexpr int TM_COLS = 512;                     // 2 buffers x NA accumulators x 64 columns <= 512
    static_assert(2 * NA * kBN <= TM_COLS, "accumulators do not fit TMEM");
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char *smem = reinterpret_cast<unsigned char *>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    unsigned char *sA = smem;                                  // NA tiles
    unsigned char *sB = sA + NA * A_TILE;                      // kBStages tiles
    uint64_t *bars = reinterpret_cast<uint64_t *>(sB + kBStages * B_TILE);
    uint64_t *b_full = bars, *b_empty = bars + kBStages;
    uint64_t *a_full = bars + 2 * kBStages, *a_empty = a_full + 1;
    uint64_t *t_full = a_empty + 1, *t_empty = t_full + 2;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(t_empty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < kBStages; ++s) { mbar_init(b_full + s, 1); mbar_init(b_empty + s, 1); }
        mbar_init(a_full, 1);
        mbar_init(a_empty, 1);
        for (int b = 0; b < 2; ++b) { mbar_init(t_full + b, 1); mbar_init(t_empty + b, kEpiWarps); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {   // TMEM: the whole 512 columns (one CTA per SM)
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    const int n_my_groups = ((int)p.n_groups - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

    if (warp == 0) {
        // ===== producer: one lane streams A tiles (per user group) and B tiles (per step) =====
        if (lane == 0) {
            uint32_t bt = 0;   // B tiles issued so far (ring position + parity)
            for (int gi = 0; gi < n_my_groups; ++gi) {
                const int64_t grp = (int64_t)blockIdx.x + (int64_t)gi * gridDim.x;
                if (gi > 0) mbar_wait(a_empty, (gi - 1) & 1);    // MMAs of the previous group are done
                mbar_expect_tx(a_full, NA * A_TILE);
                for (int a = 0; a < NA; ++a)
                    for (int kb = 0; kb < KB; ++kb)
                        bulk_g2s(sA + a * A_TILE + kb * 16384,
                                 reinterpret_cast<const unsigned char *>(p.A) + ((size_t)(grp * NA + a) * KB + kb) * 16384,
                                 16384, a_full);
                for (int j = 0; j < p.n_btiles; ++j, ++bt) {
                    const uint32_t s = bt % kBStages;
                    if (bt >= (uint32_t)kBStages) mbar_wait(b_empty + s, ((bt / kBStages) - 1) & 1);
                    mbar_expect_tx(b_full + s, B_TILE);
                    bulk_g2s(sB + s * B_TILE, reinterpret_cast<const unsigned char *>(p.B) + (size_t)j * B_TILE,
                             B_TILE, b_full + s);
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: one lane =====
        if (lane == 0) {
            uint32_t bt = 0;
            for (int gi = 0; gi < n_my_groups; ++gi) {
                mbar_wait(a_full, gi & 1);
                for (int j = 0; j < p.n_btiles; ++j, ++bt) {
                    const uint32_t s = bt % kBStages, buf = bt & 1;
                    mbar_wait(b_full + s, (bt / kBStages) & 1);
                    if (bt >= 2) mbar_wait(t_empty + buf, ((bt >> 1) - 1) & 1);   // epilogue drained this buffer
                    tc_fence_after();
#pragma unroll
                    for (int a = 0; a < NA; ++a) {
                        const uint32_t d = tmem_base + buf * (NA * kBN) + a * kBN;
#pragma unroll
                        for (int kb = 0; kb < KB; ++kb) {
                            const uint32_t abase = smem_u32(sA + a * A_TILE + kb * 16384);
                            const uint32_t bbase = smem_u32(sB + s * B_TILE + kb * (kBN * 128));
#pragma unroll
                            for (int kk = 0; kk < 4; ++kk)   // UMMA K = 16 bf16 = 32 bytes inside the swizzle atom
                                umma_bf16(d, umma_desc(abase + kk * 32), umma_desc(bbase + kk * 32), kIdesc,
                                          (kb | kk) ? 1u : 0u);
                        }
                    }
                    umma_commit(b_empty + s);     // the B stage is free once these MMAs have read it
                    umma_commit(t_full + buf);    // ... and the accumulators are complete
                }
                umma_commit(a_empty);             // A tiles may be overwritten
            }
        }
    } else {
        // ===== epilogue: warp e handles TMEM lanes 32 * (warp % 4) .. + 31 (hardware restriction:
        // a warp reaches only its own quarter) of accumulators a = (e / 4) * NA/2 .. + NA/2 - 1
        const int e = warp - 2;
        const int quarter = warp & 3;
        constexpr int NACC = NA / 2;
        const int a0 = (e >> 2) * NACC;
        uint32_t bt = 0;
        for (int gi = 0; gi < n_my_groups; ++gi) {
            const int64_t grp = (int64_t)blockIdx.x + (int64_t)gi * gridDim.x;
            float tau[NACC];
            int cnt[NACC];
            int32_t *buf_ptr[NACC];
            int64_t row[NACC];
#pragma unroll
            for (int t = 0; t < NACC; ++t) {
                row[t] = (grp * NA + a0 + t) * 128 + quarter * 32 + lane;
                const bool ok = row[t] < p.n_users;
                tau[t] = ok ? p.tau[row[t]] : INFINITY;
                cnt[t] = 0;
                buf_ptr[t] = p.cand + (ok ? row[t] : 0) * kCand;
            }
            for (int j = 0; j < p.n_btiles; ++j, ++bt) {
                const uint32_t buf = bt & 1;
                mbar_wait(t_full + buf, (bt >> 1) & 1);
                tc_fence_after();
                uint32_t v[NACC][2][32];
#pragma unroll
                for (int t = 0; t < NACC; ++t) {
                    const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + buf * (NA * kBN) + (a0 + t) * kBN;
                    tmem_ld32(taddr, v[t][0]);
                    tmem_ld32(taddr + 32, v[t][1]);
                }
                tmem_ld_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(t_empty + buf);   // accumulators are in registers: hand the buffer back
                const int item0 = j * kBN;
                const int valid = min(kBN, p.nc - item0);    // < 64 only in the last tile
#pragma unroll
                for (int t = 0; t < NACC; ++t) {
                    // one compare + one predicated OR per score: a 64-bit hit mask per row and tile.
                    // (Every lane is a different user, so branching per score would diverge on
                    // almost every instruction; ~1 of 60 scores passes.)
                    uint32_t m0 = 0, m1 = 0;
#pragma unroll
                    for (int c = 0; c < 32; ++c) {
                        if (__uint_as_float(v[t][0][c]) > tau[t]) m0 |= 1u << c;
                        if (__uint_as_float(v[t][1][c]) > tau[t]) m1 |= 1u << c;
                    }
                    if (valid < kBN) {   // ragged last tile: zero-padded items do not exist
                        m0 &= valid >= 32 ? 0xffffffffu : ((1u << valid) - 1u);
                        m1 &= valid >= 64 ? 0xffffffffu : (valid > 32 ? ((1u << (valid - 32)) - 1u) : 0u);
                    }
                    // append the hits in ascending item order; a full list stops collecting
                    while (m0) {
                        const int c = __ffs(m0) - 1;
                        m0 &= m0 - 1;
                        if (cnt[t] < kCand) buf_ptr[t][cnt[t]] = item0 + c;
                        cnt[t] = min(cnt[t] + 1, kCand + 1);
                    }
                    while (m1) {
                        const int c = __ffs(m1) - 1;
                        m1 &= m1 - 1;
                        if (cnt[t] < kCand) buf_ptr[t][cnt[t]] = item0 + 32 + c;
                        cnt[t] = min(cnt[t] + 1, kCand + 1);
                    }
                }
            }
#pragma unroll
            for (int t = 0; t < NACC; ++t)
                if (row[t] < p.n_users) p.cand_cnt[row[t]] = cnt[t];
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        __syncwarp();
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TM_COLS));
    }
}

// ---- 4. finish: exact re-score, mask, sort, certify ------------------------------------------------
struct FinishParams {
    const float *P, *Q, *ib, *ub;
    const int32_t *users;        // nullable: listed user ids of the whole call
    int64_t u0;                  // first user (position in the list / id) of this batch
    int32_t n_users, nu, nc, kpad, k;
    int predictor, has_bias;
    float mu, min_rating, max_rating;
    const int32_t *cand;
    const int32_t *cand_cnt;
    const float *tau, *eps;
    const int64_t *rated_indptr;  // nullable; indexed by list position (u0 + row)
    const int32_t *rated_items;
    int32_t N;
    int32_t *out_items;          // [n_users][N]
    double *out_scores;
    int32_t *out_counts;
    int32_t *fallback;           // [n_users] 1 = not certified
};

// One CTA per user: exact fp32 score of every candidate, masks, then the top N of them in order.
//   dots    a warp per candidate, EIGHT candidates in flight: the 32 lanes read an item row with one
//           coalesced 512-byte request (a thread per candidate would touch 32 different rows per load
//           instruction); the eight partial sums are reduced together by a transposing butterfly
//           (9 shuffles for 8 sums instead of 40)
//   masks   a thread per candidate: predictor, NaN / zero / own id, look-up in the user's rated list
//           (staged in shared memory when it is short enough)
//   select  the candidates were filtered with a loose threshold (~2.2 N of them): a 256-bin histogram
//           of the scores finds the bin that holds the N-th best; only the candidates from that bin
//           upwards (N plus a few) survive, compacted in ascending item order
//   rank    by counting among the survivors (n^2 / 128 compares per thread beat a block radix sort at
//           n ~ N, need no second pass and are stable: equal scores keep ascending item order)
// (round 2: ranking ALL ~220 candidates by counting was 14 k of the kernel's 20 k warp instructions
// per user, profiles/r02m_topn_finish_full.md.)
constexpr int kRatedStage = 2048;   // rated items of the user kept in shared memory (8 KB)
constexpr int kSurv = 512;          // survivors the ranking step has room for (N <= 128)

#ifndef MFREC_FINISH_CTAS
#define MFREC_FINISH_CTAS 7   // (8 needs 64 registers: spills in the dot loop, measured 7.2 vs 6.8 ms)
#endif
__global__ void __launch_bounds__(128, MFREC_FINISH_CTAS) topn_finish_kernel(const FinishParams p)
{
    __shared__ __align__(16) float prow[256];
    __shared__ __align__(16) uint32_t keys[kCand];   // order-preserving score bits, 0 = dropped
    __shared__ float xs[kCand];                      // first the dots, then the exact x (the quantity the threshold is on)
    __shared__ int32_t rated_s[kRatedStage];
    __shared__ __align__(16) int32_t cand_s[kCand + 8];
    __shared__ __align__(16) uint32_t skeys[kSurv];  // survivors: keys and positions in the candidate list
    __shared__ int16_t spos[kSurv];
    __shared__ int hist[256];
    __shared__ int w_cnt[4];
    __shared__ float w_max[4], w_min[4];
    __shared__ int s_bin;
    __shared__ float x_nth;
    const int row = blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t pos = p.u0 + row;
    const int64_t uid = p.users ? p.users[pos] : pos;
    const int n = p.cand_cnt[row];
    const int nn = min(n, kCand);
    if (threadIdx.x == 0) { x_nth = -INFINITY; s_bin = 0; }
    for (int f = threadIdx.x; f < p.kpad; f += 128) prow[f] = p.P[uid * p.kpad + f];
    for (int j = threadIdx.x; j < 256; j += 128) hist[j] = 0;
    const int64_t ra = p.rated_indptr ? p.rated_indptr[pos] : 0, rbnd = p.rated_indptr ? p.rated_indptr[pos + 1] : 0;
    const int nrated = (rbnd - ra) > (int64_t)kRatedStage ? kRatedStage + 1 : (int)(rbnd - ra);
    const bool rated_in_smem = nrated <= kRatedStage;
    if (rated_in_smem)
        for (int j = threadIdx.x; j < nrated; j += 128) rated_s[j] = p.rated_items[ra + j];
    const int32_t *cand = p.cand + (size_t)row * kCand;
    for (int c = threadIdx.x; c < nn; c += 128) cand_s[c] = cand[c];
    if (threadIdx.x < 8 && nn > 0) cand_s[min(nn + (int)threadIdx.x, kCand + 7)] = cand[nn - 1];   // the dots read ids in eights
    __syncthreads();
    const float bu = p.ub[uid];
    // ---- dots ----------------------------------------------------------------------------------
    {
        const int nv = p.kpad / 4;   // float4 per row: 8, 16, 32 or 64 (kpad is a multiple of 32, rows zero padded)
        const float4 *pr4 = reinterpret_cast<const float4 *>(prow);
        for (int c = warp * 8; c < nn; c += 32) {
            const float4 *q[8];
            float d[8];
            const int4 id0 = *reinterpret_cast<const int4 *>(cand_s + c), id1 = *reinterpret_cast<const int4 *>(cand_s + c + 4);
            const int ids[8] = {id0.x, id0.y, id0.z, id0.w, id1.x, id1.y, id1.z, id1.w};
#pragma unroll
            for (int t = 0; t < 8; ++t) {
                q[t] = reinterpret_cast<const float4 *>(p.Q) + (size_t)(uint32_t)ids[t] * (uint32_t)nv;
                d[t] = 0.f;
            }
            for (int f = lane; f < nv; f += 32) {
                const float4 w = pr4[f];
                float4 a[8];
#pragma unroll
                for (int t = 0; t < 8; ++t) a[t] = q[t][f];
#pragma unroll
                for (int t = 0; t < 8; ++t) {
                    d[t] = fmaf(w.x, a[t].x, d[t]); d[t] = fmaf(w.y, a[t].y, d[t]);
                    d[t] = fmaf(w.z, a[t].z, d[t]); d[t] = fmaf(w.w, a[t].w, d[t]);
                }
            }
            // transposing butterfly: at offset 16 / 8 / 4 a lane keeps the half of its sums that its
            // lane bit selects and hands the other half over; offsets 2 and 1 finish the one sum left
#pragma unroll
            for (int h = 4, o = 16; h >= 1; h >>= 1, o >>= 1) {
                const bool up = (lane & o) != 0;
#pragma unroll
                for (int j = 0; j < h; ++j) {
                    const float send = up ? d[j] : d[j + h];
                    const float keep = up ? d[j + h] : d[j];
                    d[j] = keep + __shfl_xor_sync(0xffffffffu, send, o);
                }
            }
            d[0] += __shfl_xor_sync(0xffffffffu, d[0], 2);
            d[0] += __shfl_xor_sync(0xffffffffu, d[0], 1);
            const int t = lane >> 2;   // lane bits 4, 3, 2 = the candidate of this group of four lanes
            if ((lane & 3) == 0 && c + t < nn) xs[c + t] = d[0];
        }
    }
    __syncthreads();
    // ---- scores and masks: a thread per candidate ------------------------------------------------
    int valid = 0;
    float smax = -INFINITY, smin = INFINITY;
    for (int c = threadIdx.x; c < nn; c += 128) {
        const int it = cand_s[c];
        const float dot = xs[c];
        const float bi = p.ib[it];
        const float bsum = bi + bu;
        float sc;
        switch (p.predictor) {
        case MFREC_PRED_GD_RATING: sc = dot + 1.0f; break;
        case MFREC_PRED_GD_RATING_BIAS: sc = dot + (p.mu + bsum); break;
        case MFREC_PRED_KMF_LINEAR: sc = dot + bsum; break;
        case MFREC_PRED_KMF_LOGISTIC:
            sc = p.min_rating + (1.f / (1.f + expf(-(dot + bsum)))) * (p.max_rating - p.min_rating);
            break;
        case MFREC_PRED_KMF_LINEAR_NEG: sc = p.min_rating + (dot + bsum) * (p.max_rating - p.min_rating); break;
        default: sc = dot; break;
        }
        bool ok = (sc == sc) && sc != 0.f && it != (int)uid;
        if (ok && rbnd > ra) {   // binary search in the user's (ascending) rated list
            if (rated_in_smem) {
                int lo = 0, hi = nrated;
                while (lo < hi) {
                    const int mid = (lo + hi) >> 1;
                    if (rated_s[mid] < it) lo = mid + 1; else hi = mid;
                }
                ok = !(lo < nrated && rated_s[lo] == it);
            } else {
                int64_t lo = ra, hi = rbnd;
                while (lo < hi) {
                    const int64_t mid = (lo + hi) >> 1;
                    if (p.rated_items[mid] < it) lo = mid + 1; else hi = mid;
                }
                ok = !(lo < rbnd && p.rated_items[lo] == it);
            }
        }
        keys[c] = ok ? order_bits(sc) : 0u;
        xs[c] = p.has_bias ? dot + bi : dot;
        if (ok && fabsf(sc) <= 3.0e38f) {   // (an infinite score keeps its key; it only stays out of the bin range)
            valid += 1;
            smax = fmaxf(smax, sc);
            smin = fminf(smin, sc);
        } else if (ok) {
            valid += 1;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        valid += __shfl_xor_sync(0xffffffffu, valid, o);
        smax = fmaxf(smax, __shfl_xor_sync(0xffffffffu, smax, o));
        smin = fminf(smin, __shfl_xor_sync(0xffffffffu, smin, o));
    }
    if (lane == 0) { w_cnt[warp] = valid; w_max[warp] = smax; w_min[warp] = smin; }
    __syncthreads();
    const int nvalid = w_cnt[0] + w_cnt[1] + w_cnt[2] + w_cnt[3];
    smax = fmaxf(fmaxf(w_max[0], w_max[1]), fmaxf(w_max[2], w_max[3]));
    smin = fminf(fminf(w_min[0], w_min[1]), fminf(w_min[2], w_min[3]));
    // ---- select: the histogram bin of the N-th best score ------------------------------------------
    // bin(sc) is monotone in sc (finite scores; +inf -> 255, -inf -> 0), so "bin >= the N-th best's
    // bin" keeps every candidate that can be among the first N
    const float scale = (smax > smin) ? 255.99f / (smax - smin) : 0.f;
    auto bin_of = [&](float sc) { return min(255, max(0, (int)((fminf(fmaxf(sc, smin), smax) - smin) * scale))); };
    if (nvalid > p.N) {   // (block-uniform)
        for (int c = threadIdx.x; c < nn; c += 128)
            if (keys[c]) atomicAdd(&hist[bin_of(unorder_bits(keys[c]))], 1);
        __syncthreads();
        if (warp == 0) {
            int h[8], s = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) { h[j] = hist[lane * 8 + j]; s += h[j]; }
            int suf = s;   // candidates in this lane's bins and above
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_down_sync(0xffffffffu, suf, o);
                if (lane + o < 32) suf += t;
            }
            int above = suf - s;
            if (suf >= p.N && above < p.N) {   // exactly one lane
                int b = 7;
                for (; b > 0; --b) {
                    above += h[b];
                    if (above >= p.N) break;
                }
                s_bin = lane * 8 + b;
            }
        }
        __syncthreads();
    }
    const int bin_min = s_bin;   // 0 when every valid candidate is kept
    // ---- compaction in ascending item order: warp w takes a contiguous quarter of the list ----------
    const int per = ((nn + 127) >> 7) << 5;
    const int c_lo = warp * per, c_hi = min(nn, c_lo + per);
    int mine = 0;
    for (int base = c_lo; base < c_hi; base += 32) {
        const int c = base + lane;
        const bool in = c < c_hi && keys[c] && bin_of(unorder_bits(keys[c])) >= bin_min;
        mine += __popc(__ballot_sync(0xffffffffu, in));
    }
    __syncthreads();   // (w_cnt was read above by every thread)
    if (lane == 0) w_cnt[warp] = mine;
    __syncthreads();
    int off = 0;
    for (int w = 0; w < warp; ++w) off += w_cnt[w];
    const int n_surv_all = w_cnt[0] + w_cnt[1] + w_cnt[2] + w_cnt[3];
    for (int base = c_lo; base < c_hi; base += 32) {
        const int c = base + lane;
        const bool in = c < c_hi && keys[c] && bin_of(unorder_bits(keys[c])) >= bin_min;
        const uint32_t bal = __ballot_sync(0xffffffffu, in);
        const int at = off + __popc(bal & ((1u << lane) - 1u));
        if (in && at < kSurv) { skeys[at] = keys[c]; spos[at] = (int16_t)c; }
        off += __popc(bal);
    }
    const int ns = min(n_surv_all, kSurv);
    for (int c = ns + threadIdx.x; c < ((ns + 3) & ~3); c += 128) skeys[c] = 0;   // pad to a multiple of 4
    __syncthreads();
    // ---- rank among the survivors ---------------------------------------------------------------------
    const int n4 = (ns + 3) >> 2;
    const uint4 *k4 = reinterpret_cast<const uint4 *>(skeys);
    for (int c = threadIdx.x; c < ns; c += 128) {
        const uint32_t key = skeys[c];
        const int c4 = c >> 2;
        int rank = 0;
        for (int j = 0; j < c4; ++j) {           // earlier survivors (lower item id) win ties
            const uint4 kk = k4[j];
            rank += (kk.x >= key) + (kk.y >= key) + (kk.z >= key) + (kk.w >= key);
        }
        {
            const uint4 kk = k4[c4];
            const uint32_t e[4] = {kk.x, kk.y, kk.z, kk.w};
#pragma unroll
            for (int q = 0; q < 4; ++q) rank += (q < (c & 3)) ? (e[q] >= key) : (e[q] > key);
        }
        for (int j = c4 + 1; j < n4; ++j) {
            const uint4 kk = k4[j];
            rank += (kk.x > key) + (kk.y > key) + (kk.z > key) + (kk.w > key);
        }
        if (rank < p.N) {
            const int src = spos[c];
            p.out_items[(size_t)row * p.N + rank] = cand_s[src];
            p.out_scores[(size_t)row * p.N + rank] = (double)unorder_bits(key);
            if (rank == p.N - 1) x_nth = xs[src];
        }
    }
    for (int r = nvalid + threadIdx.x; r < p.N; r += 128) {   // fewer than N valid candidates: pad
        p.out_items[(size_t)row * p.N + r] = -1;
        p.out_scores[(size_t)row * p.N + r] = 0.0;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        // certificate: the N-th best exact x among the valid candidates clears tau + eps, so no
        // item below the threshold can belong to the top N (x is monotone in the score per user)
        const bool certified = n <= kCand && n_surv_all <= kSurv && nvalid >= p.N && x_nth > p.tau[row] + p.eps[row];
        p.out_counts[row] = min(nvalid, p.N);
        p.fallback[row] = certified ? 0 : 1;
    }
}

constexpr size_t sweep_smem_bytes(int KB, int NA, int ST)
{
    return (size_t)NA * KB * 16384 + (size_t)ST * KB * kBN * 128 + 256 + 1024;
}

template <int KB, int NA, int ST>
int launch_sweep(mfrec_ctx *ctx, const SweepParams &prm, int grid)
{
    const size_t smem = sweep_smem_bytes(KB, NA, ST);
    MF_CUDA(ctx, cudaFuncSetAttribute(topn_sweep_kernel<KB, NA, ST>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    topn_sweep_kernel<KB, NA, ST><<<grid, kSweepThreads, smem, ctx->stream>>>(prm);
    MF_LAUNCH_CHECK(ctx);
    return MFREC_OK;
}

// CTAs of one sweep instantiation that fit on one SM of the current device with its launch
// configuration.  Every CTA allocates all 512 TMEM columns, so a second CTA on the same SM (from
// another shard's stream, say) would wait in tcgen05.alloc until the first one finishes.
template <int KB, int NA, int ST>
int sweep_ctas_per_sm(mfrec_ctx *ctx, int *blocks)
{
    const size_t smem = sweep_smem_bytes(KB, NA, ST);
    MF_CUDA(ctx, cudaFuncSetAttribute(topn_sweep_kernel<KB, NA, ST>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    MF_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks, topn_sweep_kernel<KB, NA, ST>, kSweepThreads, smem));
    return MFREC_OK;
}

// inverse normal CDF (Acklam's rational approximation, |error| < 1.2e-9): quantile of the threshold
double inv_norm_cdf(double pr)
{
    static const double a[] = {-3.969683028665376e+01, 2.209460984245205e+02, -2.759285104469687e+02,
                               1.383577518672690e+02, -3.066479806614716e+01, 2.506628277459239e+00};
    static const double b[] = {-5.447609879822406e+01, 1.615858368580409e+02, -1.556989798598866e+02,
                               6.680131188771972e+01, -1.328068155288572e+01};
    static const double c[] = {-7.784894002430293e-03, -3.223964580411365e-01, -2.400758277161838e+00,
                               -2.549732539343734e+00, 4.374664141464968e+00, 2.938163982698783e+00};
    static const double d[] = {7.784695709041462e-03, 3.224671290700398e-01, 2.445134137142996e+00,
                               3.754408661907416e+00};
    if (pr < 0.02425) {
        const double q = sqrt(-2 * log(pr));
        return (((((c[0] * q + c[1]) * q + c[2]) * q + c[3]) * q + c[4]) * q + c[5]) /
               ((((d[0] * q + d[1]) * q + d[2]) * q + d[3]) * q + 1);
    }
    if (pr > 1 - 0.02425) return -inv_norm_cdf(1 - pr);
    const double q = pr - 0.5, r = q * q;
    return (((((a[0] * r + a[1]) * r + a[2]) * r + a[3]) * r + a[4]) * r + a[5]) * q /
           (((((b[0] * r + b[1]) * r + b[2]) * r + b[3]) * r + b[4]) * r + 1);
}

}  // namespace

extern "C" int mfrec_topn_sweep(mfrec_ctx *ctx, int predictor, int k, const double *u, const double *v,
                                int32_t ni, int32_t nu, const int32_t *users, int32_t n_users,
                                int32_t n_candidates, const int64_t *rated_indptr, const int32_t *rated_items,
                                double mu, const double *items_bias, const double *users_bias,
                                double min_rating, double max_rating, int32_t N, int32_t *out_items,
                                double *out_scores, int32_t *out_counts, double stats[8])
{
    if (!ctx || !u || !v) return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_topn_sweep: NULL argument");
    mfrec_model *M = nullptr;
    MF_TRY(mfrec_model_create(ctx, nullptr, k, ni, nu, u, v, items_bias, users_bias, &M));
    const int rc = mfrec_model_topn_sweep(ctx, M, predictor, users, n_users, n_candidates, rated_indptr, rated_items,
                                          mu, min_rating, max_rating, N, out_items, out_scores, out_counts, stats);
    mfrec_model_destroy(M);
    return rc;
}

namespace {

// Which path a top-N call takes: the rule below (kPathAuto), or the one a multi-shard call chose for
// the whole user list (a share of it may be smaller than the rule's 128 users).
enum TopnPath { kPathAuto = 0, kPathSweep = 1, kPathExact = 2 };

// The threshold filter pays off only when the top N is a thin slice of the candidates and the
// candidate list has room for ~3N entries; everything else goes to the exact path.
bool sweep_applies(int predictor, int k, int32_t N, int32_t n_candidates, int64_t n_users)
{
    const bool has_bias = predictor != MFREC_PRED_GD_RATING && predictor != MFREC_PRED_DOT;
    const int KB = (k + (has_bias ? 1 : 0) + 63) / 64;
    return !(8 * N > kCand || (int64_t)N * 16 > n_candidates || KB > 4 || n_users < 128);
}

int topn_sweep_on_model(mfrec_ctx *ctx, const mfrec_model *M, int predictor, const int32_t *users, int32_t n_users,
                        int32_t n_candidates, const int64_t *rated_indptr, const int32_t *rated_items, double mu,
                        double min_rating, double max_rating, int32_t N, int32_t *out_items, double *out_scores,
                        int32_t *out_counts, double stats[8], int path)
{
    if (!ctx || !M || !out_items || !out_scores || !out_counts)
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_topn_sweep: NULL argument");
    if (M->user_perm || M->item_perm)
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_topn_sweep: the model must be in identity layout (created without a ratings layout)");
    const int k = M->k;
    const int32_t ni = M->ni, nu = M->nu;
    if (predictor < 0 || predictor > MFREC_PRED_DOT || n_users < 0 || N <= 0 || n_candidates < 0 || n_candidates > ni)
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_topn_sweep: predictor=%d n_users=%d N=%d n_candidates=%d",
                               predictor, n_users, N, n_candidates);
    if (users)
        for (int32_t j = 0; j < n_users; ++j)
            if (users[j] < 0 || users[j] >= nu)
                return mfrec_set_error(ctx, MFREC_ERR_INDEX, "mfrec_topn_sweep: user %d outside [0,%d)", users[j], nu);
    if (!users && n_users > nu)
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_topn_sweep: n_users=%d > nu=%d", n_users, nu);
    if (stats) memset(stats, 0, 8 * sizeof(double));
    if (n_users == 0) return MFREC_OK;
    const bool has_bias = predictor != MFREC_PRED_GD_RATING && predictor != MFREC_PRED_DOT;
    const int ka = k + (has_bias ? 1 : 0);
    const int KB = (ka + 63) / 64;
    if (path == kPathExact || (path == kPathAuto && !sweep_applies(predictor, k, N, n_candidates, n_users))) {
        std::vector<int32_t> all;
        if (!users) {
            all.resize(n_users);
            for (int32_t j = 0; j < n_users; ++j) all[j] = j;
        }
        return mfrec_topn_on_model(ctx, M, predictor, users ? users : all.data(), n_users, n_candidates, rated_indptr,
                                rated_items, mu, min_rating, max_rating, N, out_items, out_scores, out_counts, ni, nu);
    }
    MF_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    Tracer tr("topn_sweep", st);
    const int kpad = M->kpad;
    const int nc = n_candidates;
    const int NA = KB >= 3 ? 2 : 4;
    const int group = NA * 128;
    const int n_btiles = (nc + kBN - 1) / kBN;
    const int batch = (int)std::min<int64_t>((int64_t)group * ctx->sm_count, ((int64_t)n_users + group - 1) / group * group);

    // ---- moments + item operand ----------------------------------------------------------
    DevBuf<double> d_sum, d_gram;
    DevBuf<float> d_qmax2, d_tau, d_eps;
    DevBuf<__nv_bfloat16> d_A, d_B;
    DevBuf<int32_t> d_cand;
    DevBuf<int32_t> d_cnt, d_users, d_rated, d_items, d_counts, d_fb;
    DevBuf<int64_t> d_indptr;
    DevBuf<double> d_scores;
    MF_CUDA(ctx, d_sum.alloc(ka, ctx->stream));
    MF_CUDA(ctx, d_gram.alloc((size_t)ka * ka, ctx->stream));
    MF_CUDA(ctx, d_qmax2.alloc(1, ctx->stream));
    MF_CUDA(ctx, d_tau.alloc(batch, ctx->stream));
    MF_CUDA(ctx, d_eps.alloc(batch, ctx->stream));
    MF_CUDA(ctx, d_A.alloc((size_t)batch * KB * 64, ctx->stream));
    MF_CUDA(ctx, d_B.alloc((size_t)n_btiles * KB * kBN * 64, ctx->stream));
    MF_CUDA(ctx, d_cand.alloc((size_t)batch * kCand, ctx->stream));
    MF_CUDA(ctx, d_cnt.alloc(batch, ctx->stream));
    MF_CUDA(ctx, d_items.alloc((size_t)batch * N, ctx->stream));
    MF_CUDA(ctx, d_scores.alloc((size_t)batch * N, ctx->stream));
    MF_CUDA(ctx, d_counts.alloc(batch, ctx->stream));
    MF_CUDA(ctx, d_fb.alloc(batch, ctx->stream));
    if (users) {
        MF_CUDA(ctx, d_users.alloc(n_users, ctx->stream));
        MF_CUDA(ctx, cudaMemcpyAsync(d_users.p, users, (size_t)n_users * 4, cudaMemcpyHostToDevice, st));
    }
    const int64_t n_rated = rated_indptr ? rated_indptr[n_users] : 0;
    if (rated_indptr && n_rated > 0) {
        if (!rated_items) return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_topn_sweep: rated_items is NULL");
        MF_CUDA(ctx, d_indptr.alloc((size_t)n_users + 1, ctx->stream));
        MF_CUDA(ctx, d_rated.alloc((size_t)n_rated, ctx->stream));
        MF_CUDA(ctx, cudaMemcpyAsync(d_indptr.p, rated_indptr, ((size_t)n_users + 1) * 8, cudaMemcpyHostToDevice, st));
        MF_CUDA(ctx, cudaMemcpyAsync(d_rated.p, rated_items, (size_t)n_rated * 4, cudaMemcpyHostToDevice, st));
    }
    item_moments_kernel<<<dim3(ka, ka), 256, 0, st>>>(M->Q, M->ib, kpad, ka, k, nc, d_sum.p, d_gram.p, d_qmax2.p);
    MF_LAUNCH_CHECK(ctx);
    // the per-user thresholds hold the covariance in shared memory where it fits, else read it through L2
    const size_t smem_thr = ((size_t)ka * (ka | 1) + ka) * 4;
    const bool thr_in_l2 = smem_thr > ctx->smem_optin;
    DevBuf<float> d_cov;
    if (thr_in_l2) {
        MF_CUDA(ctx, d_cov.alloc((size_t)ka * ka, ctx->stream));
        item_cov_kernel<<<(ka * ka + 255) / 256, 256, 0, st>>>(d_sum.p, d_gram.p, ka, nc, d_cov.p);
        MF_LAUNCH_CHECK(ctx);
    }
    {
        const int64_t chunks = (int64_t)n_btiles * KB * kBN * 8;
        pack_operand_kernel<kBN><<<(unsigned)ceil_div64(chunks, 256), 256, 0, st>>>(
            M->Q, kpad, k, nullptr, 0, nc, nc, KB, has_bias ? k : -1, M->ib, d_B.p, chunks);
        MF_LAUNCH_CHECK(ctx);
    }
    // expected 2.2 N items above the threshold (normal approximation of a user's scores).  The
    // finish kernel's time is proportional to the candidates (it is bound by the L2 -> SM traffic
    // of their item rows, ~6 TB/s), a user with fewer than N of them is redone by the exact path:
    // measured at Netflix shape, budget 2.5 -> 12.3 ms / 0 redone, 2.1 -> 10.0 ms / 0, 1.8 ->
    // 8.5 ms / 151 users, 1.5 -> 7.2 ms / 60,785 users.
    constexpr double budget = 2.2;
    const float z = (float)inv_norm_cdf(1.0 - std::min(0.45, budget * N / (double)nc));
    tr.lap("upload + moments + pack V");

    cudaEvent_t ev[5];
    for (int j = 0; j < 5; ++j) MF_CUDA(ctx, cudaEventCreate(&ev[j]));
    double sweep_ms = 0.0, prep_ms = 0.0, finish_ms = 0.0, d2h_ms = 0.0, n_fallback = 0.0, n_cand = 0.0, n_overflow = 0.0;
    std::vector<int32_t> h_fb(batch), h_cnt(batch), fb_users;
    std::vector<int64_t> fb_pos;
    int rc = MFREC_OK;
    for (int64_t first = 0; first < n_users && rc == MFREC_OK; first += batch) {
        const int nub = (int)std::min<int64_t>(batch, n_users - first);
        const int n_groups = (nub + group - 1) / group;
        cudaEventRecord(ev[2], st);
        if (thr_in_l2) {
            user_threshold_l2_kernel<<<(nub + 7) / 8, 256, 0, st>>>(M->P, kpad, k, ka, users ? d_users.p : nullptr, first,
                                                                    nub, nu, d_sum.p, d_cov.p, d_qmax2.p, nc, z,
                                                                    d_tau.p, d_eps.p);
        } else {
            if (smem_thr > 48 * 1024)
                cudaFuncSetAttribute(user_threshold_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_thr);
            user_threshold_kernel<<<(nub + 7) / 8, 256, smem_thr, st>>>(M->P, kpad, k, ka, users ? d_users.p : nullptr, first,
                                                                       nub, nu, d_sum.p, d_gram.p, d_qmax2.p, nc, z,
                                                                       d_tau.p, d_eps.p);
        }
        MF_LAUNCH_CHECK(ctx);
        {
            const int64_t chunks = (int64_t)n_groups * NA * KB * 128 * 8;
            pack_operand_kernel<128><<<(unsigned)ceil_div64(chunks, 256), 256, 0, st>>>(
                M->P, kpad, k, users ? d_users.p : nullptr, first, nub, nu, KB, has_bias ? k : -1, nullptr, d_A.p, chunks);
            MF_LAUNCH_CHECK(ctx);
        }
        SweepParams sp;
        sp.A = d_A.p; sp.B = d_B.p; sp.tau = d_tau.p; sp.cand = d_cand.p; sp.cand_cnt = d_cnt.p;
        sp.n_users = nub; sp.n_groups = n_groups; sp.n_btiles = n_btiles; sp.nc = nc;
        const int grid = std::min(n_groups, ctx->sm_count);
        cudaEventRecord(ev[0], st);
        if (KB == 1) rc = launch_sweep<1, 4, 4>(ctx, sp, grid);
        else if (KB == 2) rc = launch_sweep<2, 4, 4>(ctx, sp, grid);
        else if (KB == 3) rc = launch_sweep<3, 2, 4>(ctx, sp, grid);
        else rc = launch_sweep<4, 2, 2>(ctx, sp, grid);
        cudaEventRecord(ev[1], st);
        if (rc != MFREC_OK) break;
        FinishParams fp;
        fp.P = M->P; fp.Q = M->Q; fp.ib = M->ib; fp.ub = M->ub;
        fp.users = users ? d_users.p : nullptr; fp.u0 = first; fp.n_users = nub; fp.nu = nu; fp.nc = nc;
        fp.kpad = kpad; fp.k = k; fp.predictor = predictor; fp.has_bias = has_bias ? 1 : 0;
        fp.mu = (float)mu; fp.min_rating = (float)min_rating; fp.max_rating = (float)max_rating;
        fp.cand = d_cand.p; fp.cand_cnt = d_cnt.p; fp.tau = d_tau.p; fp.eps = d_eps.p;
        fp.rated_indptr = d_indptr.p; fp.rated_items = d_rated.p; fp.N = N;
        fp.out_items = d_items.p; fp.out_scores = d_scores.p; fp.out_counts = d_counts.p; fp.fallback = d_fb.p;
        topn_finish_kernel<<<nub, 128, 0, st>>>(fp);
        MF_LAUNCH_CHECK(ctx);
        cudaEventRecord(ev[3], st);
        MF_CUDA(ctx, cudaMemcpyAsync(out_items + (size_t)first * N, d_items.p, (size_t)nub * N * 4, cudaMemcpyDeviceToHost, st));
        MF_CUDA(ctx, cudaMemcpyAsync(out_scores + (size_t)first * N, d_scores.p, (size_t)nub * N * 8, cudaMemcpyDeviceToHost, st));
        MF_CUDA(ctx, cudaMemcpyAsync(out_counts + first, d_counts.p, (size_t)nub * 4, cudaMemcpyDeviceToHost, st));
        MF_CUDA(ctx, cudaMemcpyAsync(h_fb.data(), d_fb.p, (size_t)nub * 4, cudaMemcpyDeviceToHost, st));
        MF_CUDA(ctx, cudaMemcpyAsync(h_cnt.data(), d_cnt.p, (size_t)nub * 4, cudaMemcpyDeviceToHost, st));
        cudaEventRecord(ev[4], st);
        MF_CUDA(ctx, cudaStreamSynchronize(st));
        float ms = 0.f;
        cudaEventElapsedTime(&ms, ev[0], ev[1]);
        sweep_ms += ms;
        cudaEventElapsedTime(&ms, ev[2], ev[0]);
        prep_ms += ms;
        cudaEventElapsedTime(&ms, ev[1], ev[3]);
        finish_ms += ms;
        cudaEventElapsedTime(&ms, ev[3], ev[4]);
        d2h_ms += ms;
        for (int j = 0; j < nub; ++j) {
            n_cand += std::min(h_cnt[j], kCand);
            if (h_cnt[j] > kCand) n_overflow += 1;
            if (h_fb[j]) {
                fb_pos.push_back(first + j);
                fb_users.push_back(users ? users[first + j] : (int32_t)(first + j));
            }
        }
    }
    for (int j = 0; j < 5; ++j) cudaEventDestroy(ev[j]);
    if (tr.on)
        fprintf(stderr, "[mfrec trace] topn_sweep: device ms: thresholds + pack U %.2f, sweep %.2f, finish %.2f, D2H %.2f\n",
                prep_ms, sweep_ms, finish_ms, d2h_ms);
    if (rc != MFREC_OK) return rc;
    tr.lap("sweep + finish");
    n_fallback = (double)fb_users.size();
    // ---- users without a certificate: exact all-items path ---------------------------------
    if (!fb_users.empty()) {
        const int32_t nf = (int32_t)fb_users.size();
        std::vector<int64_t> f_indptr(nf + 1, 0);
        std::vector<int32_t> f_rated;
        if (rated_indptr)
            for (int32_t j = 0; j < nf; ++j) {
                const int64_t a = rated_indptr[fb_pos[j]], b = rated_indptr[fb_pos[j] + 1];
                f_rated.insert(f_rated.end(), rated_items + a, rated_items + b);
                f_indptr[j + 1] = f_indptr[j] + (b - a);
            }
        std::vector<int32_t> f_items((size_t)nf * N), f_counts(nf);
        std::vector<double> f_scores((size_t)nf * N);
        MF_TRY(mfrec_topn_on_model(ctx, M, predictor, fb_users.data(), nf, n_candidates,
                                rated_indptr ? f_indptr.data() : nullptr, f_rated.empty() ? nullptr : f_rated.data(), mu,
                                min_rating, max_rating, N, f_items.data(), f_scores.data(), f_counts.data(), ni, nu));
        for (int32_t j = 0; j < nf; ++j) {
            memcpy(out_items + (size_t)fb_pos[j] * N, f_items.data() + (size_t)j * N, (size_t)N * 4);
            memcpy(out_scores + (size_t)fb_pos[j] * N, f_scores.data() + (size_t)j * N, (size_t)N * 8);
            out_counts[fb_pos[j]] = f_counts[j];
        }
        tr.lap("exact fallback");
    }
    if (stats) {
        stats[0] = n_fallback;
        stats[1] = n_cand / n_users;
        stats[2] = sweep_ms;
        stats[3] = 2.0 * (double)n_users * (double)nc * (double)k;   // useful FLOPs
        stats[4] = n_overflow;
        stats[5] = (double)KB * 64;                                   // padded K the MMAs run over
        stats[6] = z;
        stats[7] = finish_ms;
    }
    return MFREC_OK;
}

}  // namespace

extern "C" int mfrec_model_topn_sweep(mfrec_ctx *ctx, const mfrec_model *M, int predictor, const int32_t *users,
                                      int32_t n_users, int32_t n_candidates, const int64_t *rated_indptr,
                                      const int32_t *rated_items, double mu, double min_rating, double max_rating,
                                      int32_t N, int32_t *out_items, double *out_scores, int32_t *out_counts,
                                      double stats[8])
{
    return topn_sweep_on_model(ctx, M, predictor, users, n_users, n_candidates, rated_indptr, rated_items, mu,
                               min_rating, max_rating, N, out_items, out_scores, out_counts, stats, kPathAuto);
}

// A user's result depends on that user and the item side only: the moments run on a fixed (ka, ka)
// grid, z on N and n_candidates, thresholds / candidates / finish / certificate per user, and every
// uncertified user is redone alone.  The one rule that spans users is the path choice, so it is made
// here once, for the whole list, and every share takes that path whatever its size.
extern "C" int mfrec_model_topn_sweep_multi(mfrec_ctx *const *ctxs, const mfrec_model *const *models, int n_shards,
                                            int predictor, const int32_t *users, int32_t n_users, int32_t n_candidates,
                                            const int64_t *rated_indptr, const int32_t *rated_items, double mu,
                                            double min_rating, double max_rating, int32_t N, int32_t *out_items,
                                            double *out_scores, int32_t *out_counts, double stats[8])
{
    const char *who = "mfrec_model_topn_sweep_multi";
    MF_TRY(mfrec_check_shards(ctxs, models, n_shards, who));
    mfrec_ctx *ctx = ctxs[0];
    if (!out_items || !out_scores || !out_counts) return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "%s: NULL argument", who);
    for (int s = 0; s < n_shards; ++s)
        if (models[s]->user_perm || models[s]->item_perm)
            return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "%s: shard %d: the model must be in identity layout (created without a ratings layout)",
                                   who, s);
    const int k = models[0]->k;
    const int32_t ni = models[0]->ni, nu = models[0]->nu;
    if (predictor < 0 || predictor > MFREC_PRED_DOT || n_users < 0 || N <= 0 || n_candidates < 0 || n_candidates > ni)
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "%s: predictor=%d n_users=%d N=%d n_candidates=%d", who, predictor,
                               n_users, N, n_candidates);
    if (users)
        for (int32_t j = 0; j < n_users; ++j)
            if (users[j] < 0 || users[j] >= nu)
                return mfrec_set_error(ctx, MFREC_ERR_INDEX, "%s: user %d outside [0,%d)", who, users[j], nu);
    if (!users && n_users > nu) return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "%s: n_users=%d > nu=%d", who, n_users, nu);
    if (rated_indptr && n_users > 0 && rated_indptr[n_users] > 0 && !rated_items)
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "%s: rated_items is NULL", who);
    const int path = sweep_applies(predictor, k, N, n_candidates, n_users) ? kPathSweep : kPathExact;
    if (path == kPathSweep) {
        // shards on one device run at the same time: each sweep CTA takes all 512 TMEM columns, so
        // the launch configuration must keep it alone on its SM
        const bool has_bias = predictor != MFREC_PRED_GD_RATING && predictor != MFREC_PRED_DOT;
        const int KB = (k + (has_bias ? 1 : 0) + 63) / 64;
        for (int s = 0; s < n_shards; ++s) {
            MF_CUDA(ctx, cudaSetDevice(ctxs[s]->device));
            int blocks = 0;
            const int rc = KB == 1 ? sweep_ctas_per_sm<1, 4, 4>(ctx, &blocks)
                         : KB == 2 ? sweep_ctas_per_sm<2, 4, 4>(ctx, &blocks)
                         : KB == 3 ? sweep_ctas_per_sm<3, 2, 4>(ctx, &blocks)
                                   : sweep_ctas_per_sm<4, 2, 2>(ctx, &blocks);
            if (rc != MFREC_OK) return rc;
            if (blocks != 1)
                return mfrec_set_error(ctx, MFREC_ERR_UNSUPPORTED, "%s: %d sweep CTAs fit on one SM of device %d (each needs all of its tensor memory)",
                                       who, blocks, ctxs[s]->device);
        }
    }
    if (stats) memset(stats, 0, 8 * sizeof(double));
    if (n_users == 0) return MFREC_OK;

    // contiguous shares of near-equal count, cut at multiples of the 512-user sweep group where
    // every shard still gets at least one group
    constexpr int64_t kGroup = 512;
    std::vector<int64_t> cut(n_shards + 1);
    const int64_t n = n_users;
    const int64_t n_groups = (n + kGroup - 1) / kGroup;
    for (int s = 0; s <= n_shards; ++s)
        cut[s] = n >= kGroup * n_shards ? std::min(n, n_groups * s / n_shards * kGroup) : n * s / n_shards;
    std::vector<int32_t> iota;
    if (!users) {
        iota.resize(n_users);
        for (int32_t j = 0; j < n_users; ++j) iota[j] = j;
    }
    const int32_t *uid = users ? users : iota.data();
    std::vector<double> st((size_t)n_shards * 8, 0.0);
    MF_TRY(mfrec_run_shards(ctxs, n_shards, who, [&](int s) -> int {
        const int64_t a = cut[s], b = cut[s + 1];
        if (a == b) return MFREC_OK;
        // the share's rated CSR, rebased so that its indptr starts at 0
        std::vector<int64_t> ip;
        const int32_t *rated = nullptr;
        if (rated_indptr) {
            ip.resize(b - a + 1);
            for (int64_t j = 0; j <= b - a; ++j) ip[j] = rated_indptr[a + j] - rated_indptr[a];
            if (rated_items) rated = rated_items + rated_indptr[a];
        }
        return topn_sweep_on_model(ctxs[s], models[s], predictor, uid + a, (int32_t)(b - a), n_candidates,
                                   rated_indptr ? ip.data() : nullptr, rated, mu, min_rating, max_rating, N,
                                   out_items + a * N, out_scores + a * N, out_counts + a, &st[(size_t)s * 8], path);
    }));
    if (const char *path_env = getenv("MFREC_TOPN_SHARD_TIMES")) {   // debug: every shard's share and times
        if (FILE *f = fopen(path_env, "a")) {
            fprintf(f, "{\"path\": \"%s\", \"shards\": [", path == kPathSweep ? "sweep" : "exact");
            for (int s = 0; s < n_shards; ++s) {
                const double *x = &st[(size_t)s * 8];
                fprintf(f, "%s{\"device\": %d, \"users\": [%lld, %lld], \"sweep_ms\": %.4f, \"finish_ms\": %.4f, \"redone\": %.0f}",
                        s ? ", " : "", ctxs[s]->device, (long long)cut[s], (long long)cut[s + 1], x[2], x[7], x[0]);
            }
            fprintf(f, "]}\n");
            fclose(f);
        }
    }
    if (stats) {
        double cand = 0.0;
        for (int s = 0; s < n_shards; ++s) {
            const int64_t ns = cut[s + 1] - cut[s];
            if (ns == 0) continue;
            const double *x = &st[(size_t)s * 8];
            stats[0] += x[0];                          // users redone exactly
            cand += x[1] * (double)ns;                 // candidates per user, weighted by the share's users
            stats[2] = std::max(stats[2], x[2]);       // sweep ms: the slowest shard
            stats[3] += x[3];                          // useful FLOPs
            stats[4] += x[4];                          // overflowed candidate lists
            stats[5] = x[5];                           // padded K and z: the same on every shard
            stats[6] = x[6];
            stats[7] = std::max(stats[7], x[7]);       // finish ms: the slowest shard
        }
        stats[1] = cand / (double)n_users;
    }
    return MFREC_OK;
}
