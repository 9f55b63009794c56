// Alternating least squares for implicit-feedback WRMF (Hu, Koren, Volinsky, ICDM 2008):
// als_wrmf of the reference (mfrec/lib/als_implicit.pyx:208-352), driven by
// WRMFRecommender.train (mfrec/recommendation/wrmf.py:83-110).  SURVEY.md 8(f) #3 -- the step
// next to the SGD hot path, not part of it.
//
// Per epoch, with U the item factors and V the user factors (both feature-major [k][n] float64 at
// the boundary, row-major [n][k] float64 on the device):
//   user pass:  HH = sum_i u_i u_i^T ;  for every active user j with rated items S_j
//               M = HH + c_pos * sum_{i in S_j} u_i u_i^T + reg * I ,  b = (1 + c_pos) * sum_{i in S_j} u_i
//               v_j = M^-1 b                        (als_implicit.pyx:257-306)
//   item pass:  the same with the roles swapped, on the UPDATED V   (:308-352)
// Inside a pass the rows are independent, so one CTA solves one row: M is assembled in shared
// memory (k^2 doubles: k <= 165 with 227 KB per block; above that, up to k = 256, a cluster of CTAs
// shares M, see als_cluster_solve_kernel), factorised by Cholesky (M is symmetric positive definite:
// Gram matrices plus reg > 0) and solved by two triangular sweeps.  The reference inverts M with
// numpy.linalg.inv and multiplies; the two agree to float64 round-off for these well-conditioned
// systems (tests compare at 1e-9).  Everything is float64: this is a dense small-matrix problem
// at the reference's own sizes (k = 20 in its example), not a bandwidth problem.
//
// The CSR-like inputs are the reference's own (mfrec/lib/datasets.py:13-32): row = [0, count_0,
// count_1, ...] (counts, NOT offsets; the kernel loop accumulates them, als_implicit.pyx:266-268),
// col = neighbour ids in row order.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <utility>
#include <vector>

#include "common.cuh"

namespace {

constexpr int kTileMin = 8, kTileMax = 32;   // neighbour rows staged per step (as many as keep >= 4 CTAs per SM)

__global__ void __launch_bounds__(256)
to_rows_f64_kernel(const double *__restrict__ src_kn, int k, int64_t n, double *__restrict__ dst_nk)
{
    __shared__ double tile[32][33];
    const int64_t j0 = (int64_t)blockIdx.x * 32;
    const int f0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int r = ty; r < 32; r += 8) {
        const int f = f0 + r;
        const int64_t j = j0 + tx;
        tile[r][tx] = (f < k && j < n) ? src_kn[(int64_t)f * n + j] : 0.0;
    }
    __syncthreads();
    for (int r = ty; r < 32; r += 8) {
        const int64_t j = j0 + r;
        const int f = f0 + tx;
        if (j < n && f < k) dst_nk[j * k + f] = tile[tx][r];
    }
}

__global__ void __launch_bounds__(256)
from_rows_f64_kernel(const double *__restrict__ src_nk, int k, int64_t n, double *__restrict__ dst_kn)
{
    __shared__ double tile[32][33];
    const int64_t j0 = (int64_t)blockIdx.x * 32;
    const int f0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int r = ty; r < 32; r += 8) {
        const int64_t j = j0 + r;
        const int f = f0 + tx;
        tile[r][tx] = (j < n && f < k) ? src_nk[j * k + f] : 0.0;
    }
    __syncthreads();
    for (int r = ty; r < 32; r += 8) {
        const int f = f0 + r;
        const int64_t j = j0 + tx;
        if (f < k && j < n) dst_kn[(int64_t)f * n + j] = tile[tx][r];
    }
}

// partial Gram matrices: block b sums x x^T over its slice of rows, in row order
__global__ void __launch_bounds__(256)
gram_partial_kernel(const double *__restrict__ X, int64_t n, int k, int64_t rows_per_block, double *__restrict__ part)
{
    const int64_t a = (int64_t)blockIdx.x * rows_per_block, b = min(n, a + rows_per_block);
    for (int e = threadIdx.x; e < k * k; e += blockDim.x) {
        const int f1 = e / k, f2 = e % k;
        double acc = 0.0;
        for (int64_t i = a; i < b; ++i) acc += X[i * k + f1] * X[i * k + f2];
        part[(size_t)blockIdx.x * k * k + e] = acc;
    }
}

__global__ void gram_reduce_kernel(const double *__restrict__ part, int nblocks, int kk, double *__restrict__ HH)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= kk) return;
    double acc = 0.0;
    for (int b = 0; b < nblocks; ++b) acc += part[(size_t)b * kk + e];   // fixed order
    HH[e] = acc;
}

// offsets from the reference's count array: off[j] = sum_{t <= j} row[t]  (row[0] = 0)
__global__ void validate_cols_kernel(const int32_t *__restrict__ col, int64_t n, int32_t limit, int32_t *__restrict__ bad)
{
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += stride)
        if (col[j] < 0 || col[j] >= limit) atomicOr(bad, 1);
}

// one CTA per active row j: assemble M and b, Cholesky with the forward solve folded in, back
// substitution, write Y[j].  kp = the pitch of a staged neighbour row: k rounded up so that the
// register tiles below never leave the row (the padding is zero).
__host__ __device__ inline int als_pitch(int k) { return ((k + 7) / 8) * 8; }

// The solve of row j = blockIdx.x (offsets off[j], off[j + 1]); store(j, f, x) writes feature f of its
// solution.  Both instantiations (als_solve_kernel, als_solve_multi_kernel) share this code up to the store.
template <class Store>
__device__ __forceinline__ void als_solve_row(const double *__restrict__ X, const double *__restrict__ HH,
                                              const int64_t *__restrict__ off, const int32_t *__restrict__ col, int k,
                                              double c_pos, double reg, int kTile, Store store)
{
    extern __shared__ double sm[];
    const int kp = als_pitch(k);
    double *M = sm;                 // [k][k]
    double *b = M + k * k;          // [k]
    double *colv = b + k;           // [k]  column c of L during the factorisation
    double *xs = colv + k;          // [kTile][kp]
    const int j = blockIdx.x;
    const int tid = threadIdx.x, nt = blockDim.x;
    const int warp = tid >> 5, lane = tid & 31;
    for (int e = tid; e < k * k; e += nt) M[e] = HH[e];
    for (int f = tid; f < k; f += nt) b[f] = 0.0;
    for (int e = tid; e < kTile * (kp - k); e += nt) xs[(e / (kp - k)) * kp + k + e % (kp - k)] = 0.0;   // (once per row solve)
    __syncthreads();
    for (int f = tid; f < k; f += nt) M[f * k + f] += reg;
    // register tile of the Gram update: 4 rows x 8 columns of M per thread (rows ti * 4 + i, columns
    // tj + ntc * jj: neighbouring lanes read neighbouring doubles, lanes of one ti share their row
    // loads): 12 shared-memory loads per 32 multiply-adds and neighbour instead of 64 (round 1: one
    // entry per thread and step; the loop was bound by its LDS traffic and by e / k, e % k).
    const int ntr = (k + 3) / 4, ntc = kp / 8;
    const int64_t a = off[j], z = off[j + 1];
    for (int64_t t0 = a; t0 < z; t0 += kTile) {
        const int nrow = (int)min((int64_t)kTile, z - t0);
        __syncthreads();
        for (int r = warp; r < nrow; r += 4) {   // a warp copies a neighbour's row (coalesced)
            const double *src = X + (int64_t)col[t0 + r] * k;
            for (int f = lane; f < k; f += 32) xs[r * kp + f] = src[f];
        }
        __syncthreads();
        for (int tile = tid; tile < ntr * ntc; tile += nt) {
            const int ti = tile / ntc, tj = tile - ti * ntc;
            // rows past k (k not a multiple of 4) read a valid, ignored entry
            const int r0 = min(ti * 4, k - 1), r1 = min(ti * 4 + 1, k - 1), r2 = min(ti * 4 + 2, k - 1), r3 = min(ti * 4 + 3, k - 1);
            double acc[4][8];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int jj = 0; jj < 8; ++jj) acc[i][jj] = 0.0;
            const double *xr = xs;
            for (int r = 0; r < nrow; ++r, xr += kp) {
                const double rv[4] = {xr[r0], xr[r1], xr[r2], xr[r3]};
                double cv[8];
#pragma unroll
                for (int jj = 0; jj < 8; ++jj) cv[jj] = xr[tj + ntc * jj];
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int jj = 0; jj < 8; ++jj) acc[i][jj] += rv[i] * cv[jj];
            }
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int jj = 0; jj < 8; ++jj) {
                    const int f1 = ti * 4 + i, f2 = tj + ntc * jj;
                    if (f1 < k && f2 < k) M[f1 * k + f2] += c_pos * acc[i][jj];
                }
        }
        for (int f = tid; f < k; f += nt) {
            double acc = 0.0;
            for (int r = 0; r < nrow; ++r) acc += xs[r * kp + f];
            b[f] += (1.0 + c_pos) * acc;
        }
    }
    __syncthreads();
    // Cholesky M = L L^T in place (lower triangle), right-looking, two barriers per column, with the
    // forward solve L y = b riding along as one more row of the trailing update (b[r] -= L[r][c] y[c]).
    // The trailing update runs on an 8 x 16 thread grid (rows strided by 8, columns by 16: no division to
    // find an entry -- round 1 decoded (row, column) from a flat index with e / m and e % m and walked
    // the full square, 123 k of the kernel's 216 k warp instructions per row) and reads column c from
    // a contiguous copy (M[c2][c] for neighbouring c2 is one bank).
    {
        const int tr = tid >> 4, tc = tid & 15;
        for (int c = 0; c < k; ++c) {
            const double d = sqrt(M[c * k + c]);   // (every thread: the entry is final since the last barrier)
            const double yc = b[c] / d;            // y[c] (likewise)
            for (int r = c + 1 + tid; r < k; r += nt) {
                const double v = M[r * k + c] / d;
                M[r * k + c] = v;
                colv[r] = v;
            }
            __syncthreads();
            if (tid == 0) { M[c * k + c] = d; b[c] = yc; }
            for (int r = c + 1 + tr; r < k; r += 8) {
                const double lr = colv[r];
                for (int c2 = c + 1 + tc; c2 <= r; c2 += 16) M[r * k + c2] -= lr * colv[c2];
                if (tc == 15) b[r] -= lr * yc;
            }
            __syncthreads();
        }
    }
    // back substitution L^T x = y, column-oriented on one warp (row r of L is contiguous):
    // x[r] = y[r] / L[r][r], then y[c] -= L[r][c] x[r] for every c < r
    if (tid < 32) {
        for (int r = k - 1; r >= 0; --r) {
            const double xr_ = b[r] / M[r * k + r];
            for (int c = lane; c < r; c += 32) b[c] -= M[r * k + c] * xr_;
            __syncwarp();
            if (lane == 0) b[r] = xr_;
            __syncwarp();
        }
    }
    __syncthreads();
    for (int f = tid; f < k; f += nt) store(j, f, b[f]);
}

// the solved side of a multi-shard call lives once per shard: a solution goes to every copy
constexpr int kAlsMaxShards = 16;
struct AlsDst {
    double *p[kAlsMaxShards];
    int n;
};

__global__ void __launch_bounds__(128)
als_solve_kernel(const double *__restrict__ X, const double *__restrict__ HH, const int64_t *__restrict__ off,
                 const int32_t *__restrict__ col, int k, double c_pos, double reg, double *__restrict__ Y, int kTile)
{
    als_solve_row(X, HH, off, col, k, c_pos, reg, kTile, [&](int j, int f, double x) { Y[(int64_t)j * k + f] = x; });
}

// rows r0 + blockIdx.x (off / col cover this launch's rows only), stored into every copy in dst
__global__ void __launch_bounds__(128)
als_solve_multi_kernel(const double *__restrict__ X, const double *__restrict__ HH, const int64_t *__restrict__ off,
                       const int32_t *__restrict__ col, int k, double c_pos, double reg, AlsDst dst, int64_t r0, int kTile)
{
    als_solve_row(X, HH, off, col, k, c_pos, reg, kTile, [&](int j, int f, double x) {
        for (int q = 0; q < dst.n; ++q) dst.p[q][(r0 + j) * k + f] = x;
    });
}

// ---- cluster row solver: k where one CTA's shared memory cannot hold M (k > 165 at 227 KB) ----------
// One thread-block cluster of C CTAs per active row.  M lives in distributed shared memory, its rows
// dealt row-cyclically (CTA `rank` owns rows rank, rank + C, ...), so that every CTA keeps a near-equal
// share of the shrinking trailing update.  Each CTA
//   1. assembles its own rows of M = HH + c_pos * sum x x^T + reg I (lower triangle and the
//      diagonal 64-column block; nothing above is read) and its entries of b, staging every
//      neighbour row itself;
//   2. factorises M = L L^T right-looking with the forward solve L y = b riding along: for column c
//      every CTA pushes the RAW entries M[r][c] of its rows r >= c (and the owner of row c pushes
//      b[c]) into every CTA's column buffer, one cluster barrier, then every CTA derives
//      d = sqrt(M[c][c]), L[:, c] = M[:, c] / d and y[c] = b[c] / d itself -- the same operations
//      on the same operands everywhere -- and updates its own rows.  Column c + 1 of its rows is
//      updated and pushed first (look-ahead), so that the barrier's round trip overlaps the rest
//      of the trailing update.  Column buffers and the local copy of L's column alternate between
//      two slots: a CTA can be at most one column ahead of the slowest;
//   3. CTA 0 solves L^T x = y, copying L's rows out of the other CTAs' shared memory in blocks of
//      kTile rows, and writes Y[j].
// Neighbour rows are staged with coalesced loads, not bulk copies: a row is k * 8 bytes at k * 8-byte
// offsets, which the bulk copy's 16-byte rule excludes for odd k.
constexpr int kClusterThreads = 256;
constexpr int kClusterMax = 8;   // portable cluster size

__device__ __forceinline__ uint32_t cluster_ctarank()
{
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
// generic address of the same shared-memory location in CTA `rank` of the cluster
__device__ __forceinline__ double *cluster_map(double *p, uint32_t rank)
{
    uint64_t q;
    asm volatile("mapa.u64 %0, %1, %2;" : "=l"(q) : "l"(p), "r"(rank));
    return reinterpret_cast<double *>(q);
}

// staged-row pitch: whole 64-column blocks of the Gram tiles (the padding is zero)
__host__ __device__ inline int als_cluster_pitch(int k) { return ((k + 63) / 64) * 64; }
// shared memory per CTA: own rows of M [nr][k], b [nr], column buffers [2][k + 1], L's column [2][k],
// y [k], staged rows [kTile][pitch]
__host__ __device__ inline size_t als_cluster_smem(int k, int C, int kTile)
{
    const size_t nr = (size_t)(k + C - 1) / C;
    return (nr * k + nr + 2 * (size_t)(k + 1) + 2 * (size_t)k + k + (size_t)kTile * als_cluster_pitch(k)) * sizeof(double);
}

// the cluster's solve of row j = blockIdx.x / C; CTA 0 calls store(j, f, x) for every feature f of the solution
template <class Store>
__device__ __forceinline__ void als_cluster_solve_row(const double *__restrict__ X, const double *__restrict__ HH,
                                                      const int64_t *__restrict__ off, const int32_t *__restrict__ col,
                                                      int k, double c_pos, double reg, int kTile, int C, Store store)
{
    extern __shared__ double sm[];
    const int tid = threadIdx.x, nt = blockDim.x;
    const int warp = tid >> 5, lane = tid & 31, nwarp = nt >> 5;
    const int rank = (int)cluster_ctarank();
    const int nr = (k + C - 1) / C;
    const int nloc = (k - rank + C - 1) / C;   // own rows: i = rank + C * li, li < nloc
    const int kp = als_cluster_pitch(k);
    double *Ml = sm;                       // [nr][k]
    double *bl = Ml + (size_t)nr * k;      // [nr]
    double *colb = bl + nr;                // [2][k + 1]: raw M[:, c] by global row, raw b[c] at [k]
    double *lcol = colb + 2 * (k + 1);     // [2][k]: L[:, c]
    double *yv = lcol + 2 * k;             // [k]: y, then x
    double *xs = yv + k;                   // [kTile][kp]: staged neighbour rows; rows of L in step 3
    const int64_t j = blockIdx.x / C;
    cluster_arrive();   // (waited for before the first push: every CTA of the cluster is running)

    // 1. assembly
    for (int e = tid; e < nloc * k; e += nt) {
        const int li = e / k, c = e - li * k, i = rank + C * li;
        double h = HH[(size_t)i * k + c];
        if (c == i) h += reg;
        Ml[e] = h;
    }
    for (int li = tid; li < nr; li += nt) bl[li] = 0.0;
    for (int e = tid; e < kTile * (kp - k); e += nt) xs[(e / (kp - k)) * kp + k + e % (kp - k)] = 0.0;
    // register tile: 4 own rows x 8 columns (c0 + 8 jj) of one 64-column block; blocks right of the
    // tile's last row are skipped
    const int ngr = (nloc + 3) / 4, ncb = kp / 64, ntile = ngr * ncb * 8;
    const int64_t a = off[j], z = off[j + 1];
    for (int64_t t0 = a; t0 < z; t0 += kTile) {
        const int nrow = (int)min((int64_t)kTile, z - t0);
        __syncthreads();
        for (int r = warp; r < nrow; r += nwarp) {
            const double *src = X + (int64_t)col[t0 + r] * k;
            for (int f = lane; f < k; f += 32) xs[r * kp + f] = src[f];
        }
        __syncthreads();
        for (int w = tid; w < ntile; w += nt) {
            const int p = w >> 3, g = p / ncb, cb = p - g * ncb;
            if (64 * cb > rank + C * min(4 * g + 3, nloc - 1)) continue;
            const int c0 = 64 * cb + (w & 7);
            int ri[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) ri[q] = rank + C * min(4 * g + q, nloc - 1);   // (past nloc: read, ignored)
            double acc[4][8];
#pragma unroll
            for (int q = 0; q < 4; ++q)
#pragma unroll
                for (int jj = 0; jj < 8; ++jj) acc[q][jj] = 0.0;
            const double *xr = xs;
            for (int r = 0; r < nrow; ++r, xr += kp) {
                double rv[4], cv[8];
#pragma unroll
                for (int q = 0; q < 4; ++q) rv[q] = xr[ri[q]];
#pragma unroll
                for (int jj = 0; jj < 8; ++jj) cv[jj] = xr[c0 + 8 * jj];
#pragma unroll
                for (int q = 0; q < 4; ++q)
#pragma unroll
                    for (int jj = 0; jj < 8; ++jj) acc[q][jj] += rv[q] * cv[jj];
            }
#pragma unroll
            for (int q = 0; q < 4; ++q)
#pragma unroll
                for (int jj = 0; jj < 8; ++jj) {
                    const int li = 4 * g + q, c = c0 + 8 * jj;
                    if (li < nloc && c < k) Ml[li * k + c] += c_pos * acc[q][jj];
                }
        }
        for (int li = tid; li < nloc; li += nt) {
            const int i = rank + C * li;
            double acc = 0.0;
            for (int r = 0; r < nrow; ++r) acc += xs[r * kp + i];
            bl[li] += (1.0 + c_pos) * acc;
        }
    }
    __syncthreads();

    // 2. factorisation + forward solve
    cluster_wait();
    for (int li = tid; li < nloc; li += nt) {   // raw column 0
        const int i = rank + C * li;
        for (int q = 0; q < C; ++q) {
            double *dst = cluster_map(colb, q);
            dst[i] = Ml[li * k];
            if (i == 0) dst[k] = bl[li];
        }
    }
    cluster_arrive();
    const int tr = tid >> 4, tc = tid & 15;   // 16 x 16 grid of the trailing update
    for (int c = 0; c < k; ++c) {
        cluster_wait();
        const double *cb = colb + (c & 1) * (k + 1);
        double *lc = lcol + (c & 1) * k;
        const double d = sqrt(cb[c]);
        const double yc = cb[k] / d;
        for (int r = c + 1 + tid; r < k; r += nt) {
            const double v = cb[r] / d;
            lc[r] = v;
            if (r % C == rank) Ml[(r / C) * k + c] = v;
        }
        if (tid == 0) {
            yv[c] = yc;
            if (c % C == rank) Ml[(c / C) * k + c] = d;
        }
        __syncthreads();
        const int lb = c + 1 <= rank ? 0 : (c + 1 - rank + C - 1) / C;   // first own row > c
        if (c + 1 < k) {   // look-ahead: column c + 1 of the own rows, pushed to every CTA
            double *nb = colb + ((c + 1) & 1) * (k + 1);
            const double lnext = lc[c + 1];
            for (int li = lb + tid; li < nloc; li += nt) {
                const int i = rank + C * li;
                const double v = Ml[li * k + c + 1] - lc[i] * lnext;
                Ml[li * k + c + 1] = v;
                double bv = 0.0;
                if (i == c + 1) bl[li] = bv = bl[li] - lc[i] * yc;
                for (int q = 0; q < C; ++q) {
                    double *dst = cluster_map(nb, q);
                    dst[i] = v;
                    if (i == c + 1) dst[k] = bv;
                }
            }
            cluster_arrive();
        }
        for (int li = lb + tr; li < nloc; li += 16) {   // the rest: columns c + 2 .. i, b of rows > c + 1
            const int i = rank + C * li;
            const double lr = lc[i];
            for (int c2 = c + 2 + tc; c2 <= i; c2 += 16) Ml[li * k + c2] -= lr * lc[c2];
            if (tc == 15 && i > c + 1) bl[li] -= lr * yc;
        }
    }
    cluster_arrive();   // L complete in every CTA
    cluster_wait();

    // 3. back substitution L^T x = y on CTA 0, as in als_solve_kernel, kTile rows of L at a time
    if (rank == 0) {
        for (int r1 = k - 1; r1 >= 0; r1 -= kTile) {
            const int r0 = max(0, r1 - kTile + 1);
            for (int r = r0 + warp; r <= r1; r += nwarp) {
                const double *src = cluster_map(Ml + (size_t)(r / C) * k, r % C);
#pragma unroll 4
                for (int f = lane; f <= r; f += 32) xs[(r - r0) * kp + f] = src[f];
            }
            __syncthreads();
            if (tid < 32) {
                for (int r = r1; r >= r0; --r) {
                    const double *Lr = xs + (r - r0) * kp;
                    const double x = yv[r] / Lr[r];
                    for (int c = lane; c < r; c += 32) yv[c] -= Lr[c] * x;
                    __syncwarp();
                    if (lane == 0) yv[r] = x;
                    __syncwarp();
                }
            }
            __syncthreads();
        }
        for (int f = tid; f < k; f += nt) store(j, f, yv[f]);
    }
    cluster_arrive();   // the other CTAs keep their shared memory until CTA 0 has read it
    cluster_wait();
}

__global__ void __launch_bounds__(kClusterThreads, 1)
als_cluster_solve_kernel(const double *__restrict__ X, const double *__restrict__ HH, const int64_t *__restrict__ off,
                         const int32_t *__restrict__ col, int k, double c_pos, double reg, double *__restrict__ Y,
                         int kTile, int C)
{
    als_cluster_solve_row(X, HH, off, col, k, c_pos, reg, kTile, C, [&](int64_t j, int f, double x) { Y[j * k + f] = x; });
}

// rows r0 + blockIdx.x / C (off / col cover this launch's rows only), stored into every copy in dst
__global__ void __launch_bounds__(kClusterThreads, 1)
als_cluster_solve_multi_kernel(const double *__restrict__ X, const double *__restrict__ HH, const int64_t *__restrict__ off,
                               const int32_t *__restrict__ col, int k, double c_pos, double reg, AlsDst dst, int64_t r0,
                               int kTile, int C)
{
    als_cluster_solve_row(X, HH, off, col, k, c_pos, reg, kTile, C, [&](int64_t j, int f, double x) {
        for (int q = 0; q < dst.n; ++q) dst.p[q][(r0 + j) * k + f] = x;
    });
}

int gram(mfrec_ctx *ctx, const double *X, int64_t n, int k, double *part, int nblocks, double *HH)
{
    const int64_t rpb = (n + nblocks - 1) / nblocks;
    gram_partial_kernel<<<nblocks, 256, 0, ctx->stream>>>(X, n, k, rpb, part);
    MF_LAUNCH_CHECK(ctx);
    gram_reduce_kernel<<<(k * k + 255) / 256, 256, 0, ctx->stream>>>(part, nblocks, k * k, HH);
    MF_LAUNCH_CHECK(ctx);
    return MFREC_OK;
}

// host: offsets of the active rows from the reference's [0, counts...] array
std::vector<int64_t> offsets_from_counts(const int32_t *row, int64_t n_row)
{
    std::vector<int64_t> off(n_row > 0 ? n_row : 1, 0);
    int64_t start = 0;
    for (int64_t j = 0; j + 1 < n_row; ++j) {
        start += row[j];                 // als_implicit.pyx:267
        off[j] = start;
        off[j + 1] = start + row[j + 1];
    }
    return off;
}

// The row solver of one device: staged neighbour rows per step, CTAs per row (1: als_solve_kernel,
// more: als_cluster_solve_kernel) and dynamic shared memory per CTA.  A function of k and the device.
struct AlsLayout {
    int kTile = kTileMax;
    int csize = 1;
    size_t smem = 0;
};

int als_layout(mfrec_ctx *ctx, int k, const char *who, AlsLayout &L)
{
    // neighbour rows per staging step: the loads of a step are one L2 round trip, so more rows per step
    // hide it better, as long as four CTAs still fit an SM
    int kTile = kTileMax;
    while (kTile > kTileMin && ((size_t)k * k + 2 * k + (size_t)kTile * als_pitch(k)) * sizeof(double) * 4 > ctx->smem_per_sm) kTile /= 2;
    size_t smem = ((size_t)k * k + 2 * k + (size_t)kTile * als_pitch(k)) * sizeof(double);
    // k where M does not fit one CTA: the cluster solver, on the fewest CTAs whose shares fit, with as
    // many staged rows as then fit
    int csize = 1;
    if (smem > ctx->smem_optin) {
        if (k > 256)
            return mfrec_set_error(ctx, MFREC_ERR_UNSUPPORTED, "%s: k=%d > 256, the library-wide limit (as mfrec_model_create)", who, k);
        cudaFuncAttributes fa;
        MF_CUDA(ctx, cudaFuncGetAttributes(&fa, als_cluster_solve_kernel));
        const size_t budget = ctx->smem_optin > fa.sharedSizeBytes ? ctx->smem_optin - fa.sharedSizeBytes : 0;
        csize = 2;
        while (csize < kClusterMax && als_cluster_smem(k, csize, kTileMin) > budget) ++csize;
        kTile = kTileMax;
        while (kTile > kTileMin && als_cluster_smem(k, csize, kTile) > budget) kTile /= 2;
        smem = als_cluster_smem(k, csize, kTile);
        if (smem > budget)
            return mfrec_set_error(ctx, MFREC_ERR_UNSUPPORTED, "%s: k=%d needs %zu B of shared memory on each of %d CTAs", who, k, smem, csize);
    }
    L.kTile = kTile;
    L.csize = csize;
    L.smem = smem;
    return MFREC_OK;
}

}  // namespace

extern "C" int mfrec_train_als_wrmf(mfrec_ctx *ctx, int nbr_epochs, int k, double *u, double *v,
                                    const int32_t *users_row, int64_t n_users_row, const int32_t *users_col,
                                    const int32_t *items_row, int64_t n_items_row, const int32_t *items_col,
                                    int32_t nbr_users, int32_t nbr_items, int c_pos, double reg)
{
    if (!ctx || !u || !v || !users_row || !items_row)
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_train_als_wrmf: NULL argument");
    if (k <= 0 || nbr_users <= 0 || nbr_items <= 0 || nbr_epochs < 0 || n_users_row < 1 || n_items_row < 1)
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_train_als_wrmf: k=%d users=%d items=%d epochs=%d", k,
                               nbr_users, nbr_items, nbr_epochs);
    const int64_t nau = n_users_row - 1, nai = n_items_row - 1;   // active rows (als_implicit.pyx:248-249)
    if (nau > nbr_users || nai > nbr_items)
        return mfrec_set_error(ctx, MFREC_ERR_INDEX, "mfrec_train_als_wrmf: more rows in the sparse structure than users / items");
    MF_CUDA(ctx, cudaSetDevice(ctx->device));
    AlsLayout lay;
    MF_TRY(als_layout(ctx, k, "mfrec_train_als_wrmf", lay));
    const int kTile = lay.kTile, csize = lay.csize;
    const size_t smem = lay.smem;
    if (nbr_epochs == 0) return MFREC_OK;
    const std::vector<int64_t> uoff = offsets_from_counts(users_row, n_users_row);
    const std::vector<int64_t> ioff = offsets_from_counts(items_row, n_items_row);
    const int64_t nuc = uoff[nau], nic = ioff[nai];
    if ((nuc > 0 && !users_col) || (nic > 0 && !items_col))
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_train_als_wrmf: NULL column array");
    for (int64_t j = 0; j < nau; ++j)
        if (uoff[j + 1] < uoff[j]) return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_train_als_wrmf: negative count");
    for (int64_t j = 0; j < nai; ++j)
        if (ioff[j + 1] < ioff[j]) return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_train_als_wrmf: negative count");
    cudaStream_t st = ctx->stream;
    const int nblocks = ctx->sm_count;
    DevBuf<double> d_stage, d_U, d_V, d_part, d_HH;
    DevBuf<int64_t> d_uoff, d_ioff;
    DevBuf<int32_t> d_ucol, d_icol, d_bad;
    const int64_t nmax = std::max<int64_t>(nbr_users, nbr_items);
    MF_CUDA(ctx, d_stage.alloc((size_t)k * nmax, ctx->stream));
    MF_CUDA(ctx, d_U.alloc((size_t)k * nbr_items, ctx->stream));
    MF_CUDA(ctx, d_V.alloc((size_t)k * nbr_users, ctx->stream));
    MF_CUDA(ctx, d_part.alloc((size_t)nblocks * k * k, ctx->stream));
    MF_CUDA(ctx, d_HH.alloc((size_t)k * k, ctx->stream));
    MF_CUDA(ctx, d_uoff.alloc(uoff.size(), ctx->stream));
    MF_CUDA(ctx, d_ioff.alloc(ioff.size(), ctx->stream));
    MF_CUDA(ctx, d_ucol.alloc(nuc, ctx->stream));
    MF_CUDA(ctx, d_icol.alloc(nic, ctx->stream));
    MF_CUDA(ctx, d_bad.alloc(1, ctx->stream));
    MF_CUDA(ctx, cudaMemsetAsync(d_bad.p, 0, 4, st));
    MF_CUDA(ctx, cudaMemcpyAsync(d_uoff.p, uoff.data(), uoff.size() * 8, cudaMemcpyHostToDevice, st));
    MF_CUDA(ctx, cudaMemcpyAsync(d_ioff.p, ioff.data(), ioff.size() * 8, cudaMemcpyHostToDevice, st));
    if (nuc) MF_CUDA(ctx, cudaMemcpyAsync(d_ucol.p, users_col, (size_t)nuc * 4, cudaMemcpyHostToDevice, st));
    if (nic) MF_CUDA(ctx, cudaMemcpyAsync(d_icol.p, items_col, (size_t)nic * 4, cudaMemcpyHostToDevice, st));
    if (nuc) { validate_cols_kernel<<<ctx->sm_count, 256, 0, st>>>(d_ucol.p, nuc, nbr_items, d_bad.p); MF_LAUNCH_CHECK(ctx); }
    if (nic) { validate_cols_kernel<<<ctx->sm_count, 256, 0, st>>>(d_icol.p, nic, nbr_users, d_bad.p); MF_LAUNCH_CHECK(ctx); }
    int32_t h_bad = 0;
    MF_CUDA(ctx, cudaMemcpyAsync(&h_bad, d_bad.p, 4, cudaMemcpyDeviceToHost, st));
    // factors: [k][n] host -> [n][k] device
    MF_CUDA(ctx, cudaMemcpyAsync(d_stage.p, u, (size_t)k * nbr_items * 8, cudaMemcpyHostToDevice, st));
    to_rows_f64_kernel<<<dim3((unsigned)ceil_div64(nbr_items, 32), (k + 31) / 32), 256, 0, st>>>(d_stage.p, k, nbr_items, d_U.p);
    MF_LAUNCH_CHECK(ctx);
    MF_CUDA(ctx, cudaStreamSynchronize(st));   // `u` is borrowed; the stage buffer is reused for v
    if (h_bad) return mfrec_set_error(ctx, MFREC_ERR_INDEX, "mfrec_train_als_wrmf: neighbour id out of range");
    MF_CUDA(ctx, cudaMemcpyAsync(d_stage.p, v, (size_t)k * nbr_users * 8, cudaMemcpyHostToDevice, st));
    to_rows_f64_kernel<<<dim3((unsigned)ceil_div64(nbr_users, 32), (k + 31) / 32), 256, 0, st>>>(d_stage.p, k, nbr_users, d_V.p);
    MF_LAUNCH_CHECK(ctx);
    cudaLaunchConfig_t ccfg = {};
    cudaLaunchAttribute cattr[1];
    if (csize == 1) {
        MF_CUDA(ctx, cudaFuncSetAttribute(als_solve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    } else {
        MF_CUDA(ctx, cudaFuncSetAttribute(als_cluster_solve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        cattr[0].id = cudaLaunchAttributeClusterDimension;
        cattr[0].val.clusterDim.x = csize;
        cattr[0].val.clusterDim.y = 1;
        cattr[0].val.clusterDim.z = 1;
        ccfg.gridDim = dim3(csize, 1, 1);
        ccfg.blockDim = dim3(kClusterThreads, 1, 1);
        ccfg.dynamicSmemBytes = smem;
        ccfg.stream = st;
        ccfg.attrs = cattr;
        ccfg.numAttrs = 1;
        int nclusters = 0;
        MF_CUDA(ctx, cudaOccupancyMaxActiveClusters(&nclusters, als_cluster_solve_kernel, &ccfg));
        if (nclusters < 1)
            return mfrec_set_error(ctx, MFREC_ERR_UNSUPPORTED, "mfrec_train_als_wrmf: k=%d: a cluster of %d CTAs with %zu B of shared memory each does not fit the device", k, csize, smem);
    }
    // one pass: every active row of Y solved against the fixed X (HH = X^T X already computed)
    auto solve = [&](const double *X, const int64_t *doff, const int32_t *dcol, int64_t rows, double *Y) -> int {
        if (rows == 0) return MFREC_OK;
        if (csize == 1) {
            als_solve_kernel<<<(unsigned)rows, 128, smem, st>>>(X, d_HH.p, doff, dcol, k, (double)c_pos, reg, Y, kTile);
        } else {
            if (rows * csize > INT32_MAX)
                return mfrec_set_error(ctx, MFREC_ERR_UNSUPPORTED, "mfrec_train_als_wrmf: %lld rows x %d CTAs exceed one grid", (long long)rows, csize);
            ccfg.gridDim = dim3((unsigned)(rows * csize), 1, 1);
            MF_CUDA(ctx, cudaLaunchKernelEx(&ccfg, als_cluster_solve_kernel, X, (const double *)d_HH.p, doff, dcol, k,
                                            (double)c_pos, reg, Y, kTile, csize));
        }
        MF_LAUNCH_CHECK(ctx);
        return MFREC_OK;
    };
    for (int e = 0; e < nbr_epochs; ++e) {
        MF_TRY(gram(ctx, d_U.p, nbr_items, k, d_part.p, nblocks, d_HH.p));
        MF_TRY(solve(d_U.p, d_uoff.p, d_ucol.p, nau, d_V.p));
        MF_TRY(gram(ctx, d_V.p, nbr_users, k, d_part.p, nblocks, d_HH.p));
        MF_TRY(solve(d_V.p, d_ioff.p, d_icol.p, nai, d_U.p));
    }
    from_rows_f64_kernel<<<dim3((unsigned)ceil_div64(nbr_users, 32), (k + 31) / 32), 256, 0, st>>>(d_V.p, k, nbr_users, d_stage.p);
    MF_LAUNCH_CHECK(ctx);
    MF_CUDA(ctx, cudaMemcpyAsync(v, d_stage.p, (size_t)k * nbr_users * 8, cudaMemcpyDeviceToHost, st));
    MF_CUDA(ctx, cudaStreamSynchronize(st));
    from_rows_f64_kernel<<<dim3((unsigned)ceil_div64(nbr_items, 32), (k + 31) / 32), 256, 0, st>>>(d_U.p, k, nbr_items, d_stage.p);
    MF_LAUNCH_CHECK(ctx);
    MF_CUDA(ctx, cudaMemcpyAsync(u, d_stage.p, (size_t)k * nbr_items * 8, cudaMemcpyDeviceToHost, st));
    MF_CUDA(ctx, cudaStreamSynchronize(st));
    return MFREC_OK;
}

// ---- mfrec_train_als_wrmf over several shards ------------------------------------------------------
// Inside a half-pass every row's system is independent, and its only shared inputs are the fixed
// side's factors and HH.  So every shard keeps a full copy of U and V, computes HH itself (the same
// gram() with the same block count: the same sums in the same order), solves a contiguous range of
// rows with the one-device code path, and stores each solution into every shard's copy of the solved
// side (peer stores over NVLink, plain stores when the copy is on its own device).  An event per
// shard separates the half-passes.  The result is the one-device result bit for bit.
namespace {

struct AlsShard {
    int device = 0;
    mfrec_ctx *ctx = nullptr;
    cudaEvent_t done = nullptr;              // recorded after each of its solves
    std::vector<cudaEvent_t> tev;            // MFREC_ALS_SHARD_TIMES: start / end of each half-pass
    int64_t u0 = 0, u1 = 0, i0 = 0, i1 = 0;  // active users [u0, u1), items [i0, i1)
    std::vector<int64_t> huoff, hioff;       // offsets of its rows, from 0
    DevBuf<double> U, V;                     // plain cudaMalloc: other devices store into them
    DevBuf<double> stage, part, HH;          // stage: shard 0 only (host layout in and out)
    DevBuf<int64_t> uoff, ioff;
    DevBuf<int32_t> ucol, icol, bad;
    int32_t h_bad = 0;

    void release()
    {
        if (!ctx) return;
        cudaSetDevice(device);
        U.release(); V.release(); stage.release(); part.release(); HH.release();
        uoff.release(); ioff.release(); ucol.release(); icol.release(); bad.release();
        if (done) cudaEventDestroy(done);
        for (cudaEvent_t e : tev) if (e) cudaEventDestroy(e);
        done = nullptr;
        tev.clear();
        mfrec_ctx_destroy(ctx);
        ctx = nullptr;
    }
};

// Owns the shards and the peer mappings this call enabled; on every exit it waits for all streams
// (a shard's kernels store into the others' copies), then frees everything and disables those mappings.
struct AlsShards {
    std::vector<AlsShard> s;
    std::vector<std::pair<int, int>> peers;   // (device, peer device)
    int caller_device = -1;                   // current device on entry, current again on exit
    explicit AlsShards(int n) : s(n)
    {
        if (cudaGetDevice(&caller_device) != cudaSuccess) caller_device = -1;
    }
    ~AlsShards()
    {
        for (AlsShard &x : s)
            if (x.ctx) {
                cudaSetDevice(x.device);
                cudaStreamSynchronize(x.ctx->stream);
            }
        for (AlsShard &x : s) x.release();
        for (const auto &p : peers) {
            cudaSetDevice(p.first);
            cudaDeviceDisablePeerAccess(p.second);
        }
        if (caller_device >= 0) cudaSetDevice(caller_device);
    }
};

// Cuts active rows [0, n) into `parts` contiguous ranges of near-equal estimated solve cost, 3 deg k^2
// + k^3 per row (the Gram update and the Cholesky, times 3): range s ends before the first row at
// which the running cost reaches (s + 1) / parts of the total.  Ranges may be empty.
std::vector<int64_t> split_rows(const std::vector<int64_t> &off, int64_t n, int k, int parts)
{
    const int64_t kk3 = 3 * (int64_t)k * k, kkk = (int64_t)k * k * k;
    std::vector<int64_t> pre((size_t)n + 1, 0);
    for (int64_t j = 0; j < n; ++j) pre[j + 1] = pre[j] + (off[j + 1] - off[j]) * kk3 + kkk;
    std::vector<int64_t> cut((size_t)parts + 1, n);
    cut[0] = 0;
    for (int s = 1; s < parts; ++s) {
        const int64_t target = pre[n] / parts * s + pre[n] % parts * s / parts;
        const int64_t c = std::lower_bound(pre.begin(), pre.end(), target) - pre.begin();
        cut[s] = std::max(cut[s - 1], std::min(c, n));
    }
    return cut;
}

}  // namespace

extern "C" int mfrec_train_als_wrmf_multi(const int32_t *devices, int n_shards, int nbr_epochs, int k,
                                          double *u, double *v,
                                          const int32_t *users_row, int64_t n_users_row, const int32_t *users_col,
                                          const int32_t *items_row, int64_t n_items_row, const int32_t *items_col,
                                          int32_t nbr_users, int32_t nbr_items, int c_pos, double reg)
{
    const char *who = "mfrec_train_als_wrmf_multi";
    if (!devices || n_shards < 1)
        return mfrec_set_error(nullptr, MFREC_ERR_BAD_ARG, "%s: no devices", who);
    if (!u || !v || !users_row || !items_row)
        return mfrec_set_error(nullptr, MFREC_ERR_BAD_ARG, "%s: NULL argument", who);
    if (k <= 0 || nbr_users <= 0 || nbr_items <= 0 || nbr_epochs < 0 || n_users_row < 1 || n_items_row < 1)
        return mfrec_set_error(nullptr, MFREC_ERR_BAD_ARG, "%s: k=%d users=%d items=%d epochs=%d", who, k,
                               nbr_users, nbr_items, nbr_epochs);
    const int64_t nau = n_users_row - 1, nai = n_items_row - 1;
    if (nau > nbr_users || nai > nbr_items)
        return mfrec_set_error(nullptr, MFREC_ERR_INDEX, "%s: more rows in the sparse structure than users / items", who);
    if (n_shards > kAlsMaxShards)
        return mfrec_set_error(nullptr, MFREC_ERR_UNSUPPORTED, "%s: %d shards, at most %d", who, n_shards, kAlsMaxShards);
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) {
        cudaGetLastError();
        return mfrec_set_error(nullptr, MFREC_ERR_CUDA, "%s: no CUDA device; this library has no CPU path", who);
    }
    for (int d = 0; d < n_shards; ++d)
        if (devices[d] < 0 || devices[d] >= count)
            return mfrec_set_error(nullptr, MFREC_ERR_BAD_ARG, "%s: device %d of %d", who, devices[d], count);
    AlsShards G(n_shards);
    std::vector<AlsShard> &S = G.s;
    for (int d = 0; d < n_shards; ++d) {
        S[d].device = devices[d];
        MF_TRY(mfrec_ctx_create(devices[d], &S[d].ctx));
    }
    // distinct devices, and every ordered pair of them must reach the other's memory
    std::vector<int> devs;
    for (int d = 0; d < n_shards; ++d)
        if (std::find(devs.begin(), devs.end(), devices[d]) == devs.end()) devs.push_back(devices[d]);
    for (int a : devs)
        for (int b : devs) {
            if (a == b) continue;
            int can = 0;
            MF_CUDA(nullptr, cudaDeviceCanAccessPeer(&can, a, b));
            if (!can) return mfrec_set_error(nullptr, MFREC_ERR_UNSUPPORTED, "%s: device %d cannot address device %d", who, a, b);
        }
    // one solver layout and one Gram block count for all shards, those of the first shard's device (and
    // of a one-device call there): bit-identity needs the same partition of every sum
    AlsLayout lay;
    MF_TRY(als_layout(S[0].ctx, k, who, lay));
    const int nblocks = S[0].ctx->sm_count;
    std::vector<cudaLaunchConfig_t> ccfg(n_shards);
    cudaLaunchAttribute cattr[1];
    cattr[0].id = cudaLaunchAttributeClusterDimension;
    cattr[0].val.clusterDim.x = lay.csize;
    cattr[0].val.clusterDim.y = 1;
    cattr[0].val.clusterDim.z = 1;
    for (int d = 0; d < n_shards; ++d) {
        mfrec_ctx *ctx = S[d].ctx;
        MF_CUDA(nullptr, cudaSetDevice(S[d].device));
        if (lay.csize == 1) {
            if (lay.smem > ctx->smem_optin)
                return mfrec_set_error(nullptr, MFREC_ERR_UNSUPPORTED, "%s: k=%d: device %d cannot give one CTA %zu B of shared memory",
                                       who, k, S[d].device, lay.smem);
            MF_CUDA(nullptr, cudaFuncSetAttribute(als_solve_multi_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lay.smem));
        } else {
            MF_CUDA(nullptr, cudaFuncSetAttribute(als_cluster_solve_multi_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lay.smem));
            cudaLaunchConfig_t &c = ccfg[d];
            c = {};
            c.gridDim = dim3(lay.csize, 1, 1);
            c.blockDim = dim3(kClusterThreads, 1, 1);
            c.dynamicSmemBytes = lay.smem;
            c.stream = ctx->stream;
            c.attrs = cattr;
            c.numAttrs = 1;
            int nclusters = 0;
            MF_CUDA(nullptr, cudaOccupancyMaxActiveClusters(&nclusters, als_cluster_solve_multi_kernel, &c));
            if (nclusters < 1)
                return mfrec_set_error(nullptr, MFREC_ERR_UNSUPPORTED, "%s: k=%d: a cluster of %d CTAs with %zu B of shared memory each does not fit device %d",
                                       who, k, lay.csize, lay.smem, S[d].device);
        }
    }
    if (nbr_epochs == 0) return MFREC_OK;
    const std::vector<int64_t> uoff = offsets_from_counts(users_row, n_users_row);
    const std::vector<int64_t> ioff = offsets_from_counts(items_row, n_items_row);
    const int64_t nuc = uoff[nau], nic = ioff[nai];
    if ((nuc > 0 && !users_col) || (nic > 0 && !items_col))
        return mfrec_set_error(nullptr, MFREC_ERR_BAD_ARG, "%s: NULL column array", who);
    for (int64_t j = 0; j < nau; ++j)
        if (uoff[j + 1] < uoff[j]) return mfrec_set_error(nullptr, MFREC_ERR_BAD_ARG, "%s: negative count", who);
    for (int64_t j = 0; j < nai; ++j)
        if (ioff[j + 1] < ioff[j]) return mfrec_set_error(nullptr, MFREC_ERR_BAD_ARG, "%s: negative count", who);
    const std::vector<int64_t> cu = split_rows(uoff, nau, k, n_shards), ci = split_rows(ioff, nai, k, n_shards);
    for (int a : devs)   // before the first launch
        for (int b : devs) {
            if (a == b) continue;
            MF_CUDA(nullptr, cudaSetDevice(a));
            const cudaError_t e = cudaDeviceEnablePeerAccess(b, 0);
            if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
            else {
                MF_CUDA(nullptr, e);
                G.peers.emplace_back(a, b);
            }
        }
    const char *times_path = getenv("MFREC_ALS_SHARD_TIMES");
    // ---- per shard: its rows' structure and the validation of their neighbour ids --------------------
    for (int d = 0; d < n_shards; ++d) {
        AlsShard &s = S[d];
        mfrec_ctx *ctx = s.ctx;
        cudaStream_t st = ctx->stream;
        MF_CUDA(nullptr, cudaSetDevice(s.device));
        s.u0 = cu[d]; s.u1 = cu[d + 1]; s.i0 = ci[d]; s.i1 = ci[d + 1];
        s.huoff.resize(s.u1 - s.u0 + 1);
        s.hioff.resize(s.i1 - s.i0 + 1);
        for (int64_t j = s.u0; j <= s.u1; ++j) s.huoff[j - s.u0] = uoff[j] - uoff[s.u0];
        for (int64_t j = s.i0; j <= s.i1; ++j) s.hioff[j - s.i0] = ioff[j] - ioff[s.i0];
        const int64_t nuc_s = s.huoff.back(), nic_s = s.hioff.back();
        MF_CUDA(nullptr, cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming));
        if (times_path) {
            s.tev.assign((size_t)4 * nbr_epochs, nullptr);
            for (cudaEvent_t &e : s.tev) MF_CUDA(nullptr, cudaEventCreate(&e));
        }
        if (d == 0) MF_CUDA(nullptr, s.stage.alloc((size_t)k * std::max<int64_t>(nbr_users, nbr_items), st));
        MF_CUDA(nullptr, s.U.alloc((size_t)k * nbr_items));
        MF_CUDA(nullptr, s.V.alloc((size_t)k * nbr_users));
        MF_CUDA(nullptr, s.part.alloc((size_t)nblocks * k * k, st));
        MF_CUDA(nullptr, s.HH.alloc((size_t)k * k, st));
        MF_CUDA(nullptr, s.uoff.alloc(s.huoff.size(), st));
        MF_CUDA(nullptr, s.ioff.alloc(s.hioff.size(), st));
        MF_CUDA(nullptr, s.ucol.alloc(nuc_s, st));
        MF_CUDA(nullptr, s.icol.alloc(nic_s, st));
        MF_CUDA(nullptr, s.bad.alloc(1, st));
        MF_CUDA(nullptr, cudaMemsetAsync(s.bad.p, 0, 4, st));
        MF_CUDA(nullptr, cudaMemcpyAsync(s.uoff.p, s.huoff.data(), s.huoff.size() * 8, cudaMemcpyHostToDevice, st));
        MF_CUDA(nullptr, cudaMemcpyAsync(s.ioff.p, s.hioff.data(), s.hioff.size() * 8, cudaMemcpyHostToDevice, st));
        if (nuc_s) MF_CUDA(nullptr, cudaMemcpyAsync(s.ucol.p, users_col + uoff[s.u0], (size_t)nuc_s * 4, cudaMemcpyHostToDevice, st));
        if (nic_s) MF_CUDA(nullptr, cudaMemcpyAsync(s.icol.p, items_col + ioff[s.i0], (size_t)nic_s * 4, cudaMemcpyHostToDevice, st));
        if (nuc_s) { validate_cols_kernel<<<ctx->sm_count, 256, 0, st>>>(s.ucol.p, nuc_s, nbr_items, s.bad.p); MF_LAUNCH_CHECK(ctx); }
        if (nic_s) { validate_cols_kernel<<<ctx->sm_count, 256, 0, st>>>(s.icol.p, nic_s, nbr_users, s.bad.p); MF_LAUNCH_CHECK(ctx); }
        MF_CUDA(nullptr, cudaMemcpyAsync(&s.h_bad, s.bad.p, 4, cudaMemcpyDeviceToHost, st));
    }
    for (int d = 0; d < n_shards; ++d) {
        MF_CUDA(nullptr, cudaSetDevice(S[d].device));
        MF_CUDA(nullptr, cudaStreamSynchronize(S[d].ctx->stream));
    }
    for (int d = 0; d < n_shards; ++d)
        if (S[d].h_bad) return mfrec_set_error(nullptr, MFREC_ERR_INDEX, "%s: neighbour id out of range", who);
    // ---- factors: [k][n] host -> [n][k] on shard 0 (one host transfer per side), then device to device
    // into every other shard's copies (over NVLink between devices)
    {
        AlsShard &s0 = S[0];
        cudaStream_t st = s0.ctx->stream;
        MF_CUDA(nullptr, cudaSetDevice(s0.device));
        MF_CUDA(nullptr, cudaMemcpyAsync(s0.stage.p, u, (size_t)k * nbr_items * 8, cudaMemcpyHostToDevice, st));
        to_rows_f64_kernel<<<dim3((unsigned)ceil_div64(nbr_items, 32), (k + 31) / 32), 256, 0, st>>>(s0.stage.p, k, nbr_items, s0.U.p);
        MF_LAUNCH_CHECK(s0.ctx);
        MF_CUDA(nullptr, cudaMemcpyAsync(s0.stage.p, v, (size_t)k * nbr_users * 8, cudaMemcpyHostToDevice, st));
        to_rows_f64_kernel<<<dim3((unsigned)ceil_div64(nbr_users, 32), (k + 31) / 32), 256, 0, st>>>(s0.stage.p, k, nbr_users, s0.V.p);
        MF_LAUNCH_CHECK(s0.ctx);
        MF_CUDA(nullptr, cudaEventRecord(s0.done, st));
    }
    for (int d = 1; d < n_shards; ++d) {   // (shard 0 overwrites its copies only after every shard's done event)
        AlsShard &s = S[d];
        cudaStream_t st = s.ctx->stream;
        MF_CUDA(nullptr, cudaSetDevice(s.device));
        MF_CUDA(nullptr, cudaStreamWaitEvent(st, S[0].done, 0));
        MF_CUDA(nullptr, cudaMemcpyPeerAsync(s.U.p, s.device, S[0].U.p, S[0].device, (size_t)k * nbr_items * 8, st));
        MF_CUDA(nullptr, cudaMemcpyPeerAsync(s.V.p, s.device, S[0].V.p, S[0].device, (size_t)k * nbr_users * 8, st));
        MF_CUDA(nullptr, cudaEventRecord(s.done, st));
    }
    // ---- half-passes ----------------------------------------------------------------------------------
    // every shard's stream first waits for every other shard's last solve (or upload): the Gram reads the
    // side they stored into, and this pass overwrites the side they read
    int hp = 0;
    auto half_pass = [&](bool users) -> int {
        for (int d = 0; d < n_shards; ++d) {
            MF_CUDA(nullptr, cudaSetDevice(S[d].device));
            for (int t = 0; t < n_shards; ++t)
                if (t != d) MF_CUDA(nullptr, cudaStreamWaitEvent(S[d].ctx->stream, S[t].done, 0));
        }
        for (int d = 0; d < n_shards; ++d) {
            AlsShard &s = S[d];
            mfrec_ctx *ctx = s.ctx;
            cudaStream_t st = ctx->stream;
            MF_CUDA(nullptr, cudaSetDevice(s.device));
            if (times_path) MF_CUDA(nullptr, cudaEventRecord(s.tev[2 * hp], st));
            const double *X = users ? s.U.p : s.V.p;
            MF_TRY(gram(ctx, X, users ? nbr_items : nbr_users, k, s.part.p, nblocks, s.HH.p));
            const int64_t r0 = users ? s.u0 : s.i0, rows = (users ? s.u1 : s.i1) - r0;
            const int64_t *doff = users ? s.uoff.p : s.ioff.p;
            const int32_t *dcol = users ? s.ucol.p : s.icol.p;
            AlsDst dst = {};
            dst.n = n_shards;
            for (int t = 0; t < n_shards; ++t) dst.p[t] = users ? S[t].V.p : S[t].U.p;
            if (rows > 0) {
                if (lay.csize == 1) {
                    als_solve_multi_kernel<<<(unsigned)rows, 128, lay.smem, st>>>(X, s.HH.p, doff, dcol, k, (double)c_pos, reg, dst, r0, lay.kTile);
                } else {
                    if (rows * lay.csize > INT32_MAX)
                        return mfrec_set_error(nullptr, MFREC_ERR_UNSUPPORTED, "%s: %lld rows x %d CTAs exceed one grid", who, (long long)rows, lay.csize);
                    ccfg[d].gridDim = dim3((unsigned)(rows * lay.csize), 1, 1);
                    MF_CUDA(nullptr, cudaLaunchKernelEx(&ccfg[d], als_cluster_solve_multi_kernel, X, (const double *)s.HH.p, doff, dcol, k,
                                                        (double)c_pos, reg, dst, r0, lay.kTile, lay.csize));
                }
                MF_LAUNCH_CHECK(ctx);
            }
            if (times_path) MF_CUDA(nullptr, cudaEventRecord(s.tev[2 * hp + 1], st));
            MF_CUDA(nullptr, cudaEventRecord(s.done, st));
        }
        ++hp;
        return MFREC_OK;
    };
    for (int e = 0; e < nbr_epochs; ++e) {
        MF_TRY(half_pass(true));
        MF_TRY(half_pass(false));
    }
    // ---- result: shard 0's copies, once every shard's last stores have landed -------------------------
    AlsShard &s0 = S[0];
    cudaStream_t st = s0.ctx->stream;
    MF_CUDA(nullptr, cudaSetDevice(s0.device));
    for (int t = 1; t < n_shards; ++t) MF_CUDA(nullptr, cudaStreamWaitEvent(st, S[t].done, 0));
    from_rows_f64_kernel<<<dim3((unsigned)ceil_div64(nbr_users, 32), (k + 31) / 32), 256, 0, st>>>(s0.V.p, k, nbr_users, s0.stage.p);
    MF_LAUNCH_CHECK(s0.ctx);
    MF_CUDA(nullptr, cudaMemcpyAsync(v, s0.stage.p, (size_t)k * nbr_users * 8, cudaMemcpyDeviceToHost, st));
    MF_CUDA(nullptr, cudaStreamSynchronize(st));
    from_rows_f64_kernel<<<dim3((unsigned)ceil_div64(nbr_items, 32), (k + 31) / 32), 256, 0, st>>>(s0.U.p, k, nbr_items, s0.stage.p);
    MF_LAUNCH_CHECK(s0.ctx);
    MF_CUDA(nullptr, cudaMemcpyAsync(u, s0.stage.p, (size_t)k * nbr_items * 8, cudaMemcpyDeviceToHost, st));
    MF_CUDA(nullptr, cudaStreamSynchronize(st));
    if (times_path) {   // one JSON line per call: each shard's rows and milliseconds per half-pass
        for (AlsShard &s : S) {
            MF_CUDA(nullptr, cudaSetDevice(s.device));
            MF_CUDA(nullptr, cudaStreamSynchronize(s.ctx->stream));
        }
        FILE *f = fopen(times_path, "a");
        if (f) {
            fprintf(f, "{\"k\": %d, \"epochs\": %d, \"csize\": %d, \"shards\": [", k, nbr_epochs, lay.csize);
            for (int d = 0; d < n_shards; ++d) {
                const AlsShard &s = S[d];
                fprintf(f, "%s{\"device\": %d, \"users\": [%lld, %lld], \"items\": [%lld, %lld], \"half_pass_ms\": [", d ? ", " : "",
                        s.device, (long long)s.u0, (long long)s.u1, (long long)s.i0, (long long)s.i1);
                for (int h = 0; h < hp; ++h) {
                    float ms = 0.f;
                    cudaEventElapsedTime(&ms, s.tev[2 * h], s.tev[2 * h + 1]);
                    fprintf(f, "%s%.4f", h ? ", " : "", ms);
                }
                fprintf(f, "]}");
            }
            fprintf(f, "]}\n");
            fclose(f);
        }
    }
    return MFREC_OK;
}
