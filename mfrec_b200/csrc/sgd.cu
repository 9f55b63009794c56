// SGD update kernels for the all-k "KMF" loops of the reference
// (mfrec/lib/kmf_train.pyx:195-277 train_linear_kernel, :103-189 train_logistic_kernel).
//
// Stratified schedule (MFREC_SCHED_STRATIFIED)
// --------------------------------------------
// Two updates commute iff they share neither the user row nor the item row.  pack.cu cuts the
// rating matrix into B x B blocks (x G item slabs) and every block into W x W buckets.
// One epoch = B sub-epochs per slab.  In sub-epoch s, CTA rb owns
//   row block rb  x  column block (rb + s) mod B            (a Latin square: no two CTAs share
//                                                            a row block or a column block)
// and inside the CTA, in phase p, warp w owns
//   row group w   x  column group (w + p) mod W             (again a Latin square)
// So at any instant all B*W warps of the grid work on pairwise disjoint users and items: no
// atomics, no locks, deterministic for a given layout.  Any serial replay that visits
// (sub-epoch, CTA, phase, warp, bucket order) nested in that order is an equivalent sequential
// SGD order; tests replay exactly that with the CPU oracle.
//
// One persistent cooperative launch runs all B sub-epochs of a slab: column blocks pass from CTA
// to CTA through release/acquire counters in global memory, column groups from warp to warp
// through counters in shared memory (see sgd_block_kernel), so there is no grid-wide or
// CTA-wide barrier on the critical path.
//
// Data movement per CTA and sub-epoch
//   * the column block's Q rows (contiguous in packed-id order) are pulled into shared memory
//     once with cp.async.bulk (TMA, mbarrier complete_tx) and written back once;
//   * each warp's W buckets are stored back to back, so the warp streams ONE contiguous run of
//     12-byte ratings through a private 4-stage shared-memory ring filled by cp.async.bulk;
//   * P rows are fetched with cp.async (16 bytes per lane, coalesced 512 B per row at k = 128)
//     into a 16-deep shared-memory ring, 16 ratings ahead of the consumer and across phase
//     boundaries; they are tracked by cp.async groups, not by the register scoreboard, so a
//     wait never stalls on the newest request; updated rows go back with 128-bit stores;
//   * the dot product's cross-lane sum is one REDUX in 32-bit fixed point; all other arithmetic
//     is fp32, the epoch's sum of squared errors is accumulated in fp64.
//
// Sequential schedule (MFREC_SCHED_SEQUENTIAL): one thread, fp64, no FMA contraction, the
// reference's exact order on the reference's own [k][n] layout.  Bit-exact with the reference
// for the linear kernel; used for verification and for tiny fold-in calls.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <thread>
#include <type_traits>

#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.cuh"
#include "fold.h"

namespace {

constexpr int kChunk = 64;    // ratings per TMA chunk
constexpr int kStages = 4;    // chunks in flight per warp (ring of kStages * kChunk ratings)
constexpr int kDepth = 16;    // P rows in flight per warp (cp.async ring), in stream positions
constexpr int kQuadsAhead = kDepth / 4;
constexpr int kRing = kChunk * kStages;
static_assert(kChunk % 4 == 0, "chunks must be 16-byte multiples");
static_assert(4 * kDepth <= kChunk, "the prefetch cursor may run at most one chunk ahead");

// Per-rank arguments.  One per launch on a real device; the ring test on ONE device passes one per
// emulated rank (CTA group g = blockIdx.x / B acts as rank g, see mfrec_ring_epochs).
struct SgdRank {
    const PackedRating *packed;
    const int64_t *bucket_off;
    const int32_t *col_start;
    float *Q, *ib, *P, *ub;   // Q / ib: this rank's copy of the item side (all slabs; only the slab in hand is current)
    double *se_part;          // [epochs of the launch][B] per-CTA sums of squared errors
    int32_t *ticks;           // [G*B] uses completed on each column block as seen by this rank, or null
                              // (null: no hand-over, the launch must cover exactly one sub-epoch)
    // ring (world > 1): where the LAST sub-epoch of a step leaves a column block -- the copy of the
    // rank that works on this slab next -- and that rank's counters
    float *peer_Q, *peer_ib;
    int32_t *peer_ticks;
    int32_t *abort;           // [1] != 0: a hand-over wait timed out somewhere, give up
    int rank;
};

struct SgdParams {
    SgdRank self;             // the arguments when ranks == null
    const SgdRank *ranks;     // device array, one per CTA group of B (ring launches only)
    // Iterations [it_begin, it_end) of the flattened (epoch, step, sub-epoch) space:
    //   it = (epoch * G + step) * B + s,   slab of a step = (rank + step) mod G
    int64_t it_begin, it_end;
    int64_t e_base;           // epoch whose sums go to se_part[0 .. B)
    int se_stride;            // doubles between two epochs' sums in se_part (B, or ranks * B in the ring test)
    int B, W, G, world;       // world > 1: slabs move around a ring of `world` = G ranks
    int tile_rows;            // shared-memory rows reserved for the Q tile
    float lr, Ku, Ki, Kb;
    int update_users, update_items;
    float fx_scale, fx_inv;       // fixed-point scale of the warp reduction (power of two)
    unsigned long long wait_ns;   // ring: give up a hand-over wait after this long (0 = never)
};

// ---- PTX helpers: cp.async (mbarrier and bulk-copy helpers: common.cuh) -------------------
template <int BYTES>
__device__ __forceinline__ void cp_async(void *dst_smem, const void *src_gmem)
{
    if constexpr (BYTES == 16)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst_smem)), "l"(src_gmem) : "memory");
    else
        asm volatile("cp.async.ca.shared.global [%0], [%1], %2;" ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "n"(BYTES) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// ---- per-lane row fragment: E floats, as NV vectors of V floats, interleaved over the warp --
template <int E>
struct Frag {
    static constexpr int V = E >= 4 ? 4 : E;
    static constexpr int NV = E / V;
    float x[E];
};

template <int E>
__device__ __forceinline__ void frag_load(Frag<E> &f, const float *row, int lane)
{
    constexpr int V = Frag<E>::V, NV = Frag<E>::NV;
#pragma unroll
    for (int c = 0; c < NV; ++c) {
        const float *p = row + (c * 32 + lane) * V;
        if constexpr (V == 4) {
            const float4 t = *reinterpret_cast<const float4 *>(p);
            f.x[c * 4 + 0] = t.x; f.x[c * 4 + 1] = t.y; f.x[c * 4 + 2] = t.z; f.x[c * 4 + 3] = t.w;
        } else if constexpr (V == 2) {
            const float2 t = *reinterpret_cast<const float2 *>(p);
            f.x[0] = t.x; f.x[1] = t.y;
        } else {
            f.x[0] = *p;
        }
    }
}

template <int E>
__device__ __forceinline__ void frag_store(const Frag<E> &f, float *row, int lane)
{
    constexpr int V = Frag<E>::V, NV = Frag<E>::NV;
#pragma unroll
    for (int c = 0; c < NV; ++c) {
        float *p = row + (c * 32 + lane) * V;
        if constexpr (V == 4)
            *reinterpret_cast<float4 *>(p) = make_float4(f.x[c * 4], f.x[c * 4 + 1], f.x[c * 4 + 2], f.x[c * 4 + 3]);
        else if constexpr (V == 2)
            *reinterpret_cast<float2 *>(p) = make_float2(f.x[0], f.x[1]);
        else
            *p = f.x[0];
    }
}

// the same with a pointer that already includes the lane's offset (row + lane * V)
template <int E>
__device__ __forceinline__ void frag_store_lane(const Frag<E> &f, float *p)
{
    constexpr int V = Frag<E>::V, NV = Frag<E>::NV;
#pragma unroll
    for (int c = 0; c < NV; ++c) {
        if constexpr (V == 4)
            *reinterpret_cast<float4 *>(p + c * 128) = make_float4(f.x[c * 4], f.x[c * 4 + 1], f.x[c * 4 + 2], f.x[c * 4 + 3]);
        else if constexpr (V == 2)
            *reinterpret_cast<float2 *>(p) = make_float2(f.x[0], f.x[1]);
        else
            *p = f.x[0];
    }
}

// base + idx * stride as ONE 64-bit multiply-add (the compiler otherwise splits the masked id into
// shifts and masks: 5-6 instructions per row address instead of 1)
template <typename T>
__device__ __forceinline__ T *row_ptr(T *base, uint32_t idx, uint32_t stride_bytes)
{
    uint64_t a;
    asm("mad.wide.u32 %0, %1, %2, %3;" : "=l"(a) : "r"(idx), "r"(stride_bytes), "l"(base));
    return reinterpret_cast<T *>(a);
}

// ---- user-factor storage (mfrec_opts.storage): P rows may live in HBM as fp16 or bf16; the
// arithmetic is fp32 either way (rows are widened on load and narrowed on store).
// fp16 narrows with round-to-nearest (11 significant bits: one SGD step moves a factor by
// ~0.3 %, i.e. several ulps).  bf16 has 8: the same step is BELOW half an ulp, round-to-nearest
// would discard most updates, so bf16 narrows with STOCHASTIC rounding (the low 16 bits plus a
// per-lane pseudo-random 16-bit number carry into the kept half): unbiased, deterministic for a
// given layout.
template <int E, typename PT>
__device__ __forceinline__ void pfrag_load(Frag<E> &f, const PT *row, int lane)
{
    if constexpr (sizeof(PT) == 4) {
        frag_load<E>(f, reinterpret_cast<const float *>(row), lane);
    } else {
        constexpr int V = Frag<E>::V, NV = Frag<E>::NV;
        static_assert(V >= 2, "16-bit rows need at least two elements per lane");
#pragma unroll
        for (int c = 0; c < NV; ++c) {
            const PT *p = row + (c * 32 + lane) * V;
#pragma unroll
            for (int h = 0; h < V / 2; ++h) {
                float2 t;
                if constexpr (std::is_same<PT, __half>::value)
                    t = __half22float2(*reinterpret_cast<const __half2 *>(p + 2 * h));
                else
                    t = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162 *>(p + 2 * h));
                f.x[c * V + 2 * h] = t.x;
                f.x[c * V + 2 * h + 1] = t.y;
            }
        }
    }
}

// p already includes the lane's offset (row + lane * V)
template <int E, typename PT>
__device__ __forceinline__ void pfrag_store_lane(const Frag<E> &f, PT *p, uint32_t &rng)
{
    if constexpr (sizeof(PT) == 4) {
        frag_store_lane<E>(f, reinterpret_cast<float *>(p));
    } else {
        constexpr int V = Frag<E>::V, NV = Frag<E>::NV;
#pragma unroll
        for (int c = 0; c < NV; ++c) {
            uint32_t w[V / 2];
#pragma unroll
            for (int h = 0; h < V / 2; ++h) {
                const float a = f.x[c * V + 2 * h], b = f.x[c * V + 2 * h + 1];
                if constexpr (std::is_same<PT, __half>::value) {
                    const __half2 t = __floats2half2_rn(a, b);
                    w[h] = *reinterpret_cast<const uint32_t *>(&t);
                } else {
                    rng = rng * 1664525u + 1013904223u;
                    const uint32_t ua = __float_as_uint(a) + (rng & 0xffffu);
                    const uint32_t ub = __float_as_uint(b) + (rng >> 16);
                    w[h] = (ua >> 16) | (ub & 0xffff0000u);
                }
            }
            PT *q = p + c * 32 * V;
            if constexpr (V == 4) *reinterpret_cast<uint2 *>(q) = make_uint2(w[0], w[1]);
            else *reinterpret_cast<uint32_t *>(q) = w[0];
        }
    }
}

// Packed fp32 pairs (sm_100: FMUL2 / FFMA2 take two independent IEEE operations per instruction;
// each half rounds exactly like the scalar instruction).  The hot loop is bound by the number of
// instructions a warp issues, so the row updates and the dot product run on pairs.
__device__ __forceinline__ unsigned long long pack2(float lo, float hi)
{
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack2(unsigned long long v, float &lo, float &hi)
{
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ unsigned long long mul2(unsigned long long a, unsigned long long b)
{
    unsigned long long r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ unsigned long long fma2(unsigned long long a, unsigned long long b, unsigned long long c)
{
    unsigned long long r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}

// system scope: the counter (and the data it guards) was written by / is read by another GPU
// (the gpu-scope pair is in common.cuh)
__device__ __forceinline__ int ld_acquire_sys(const int32_t *p)
{
    int v;
    asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(int32_t *p, int v)
{
    asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned long long global_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

// ------------------------------------------------------------------------------------------
// The stratified kernel.  grid = B CTAs (one per SM, cooperative launch), block = W warps,
// E = kpad / 32 floats per lane.  One launch runs sub-epochs [s_begin, s_end) of one item slab.
//
// CTA level: in sub-epoch s CTA rb owns column block cb = (rb + s) mod B.  Its previous owner was
// CTA rb + 1 in sub-epoch s - 1, so instead of a grid-wide barrier (a kernel boundary) between
// sub-epochs the column block is handed over through a per-block counter in global memory:
// the owner writes its Q tile back, fences, and releases ticks[cb] = s + 1; the next owner
// acquires ticks[cb] == s before it pulls the tile.  The result is the same as with one launch per
// sub-epoch (the serial replay order is unchanged), but a slow CTA only delays the two CTAs that
// depend on it, not the whole grid.
//
// Warp level: the same hand-over inside the CTA.  In phase p warp w owns column group
// (w + p) mod W, last used by warp w + 1 in phase p - 1; a shared-memory counter per warp
// replaces the CTA-wide barrier between phases.
//
// Every warp walks ONE contiguous stream of packed ratings per sub-epoch (its W buckets, stored
// back to back) with three cursors:
//   load cursor     : cp.async.bulk chunks of kChunk ratings into a kStages-deep ring
//   prefetch cursor : kDepth ratings ahead of the consumer, cp.async of the P row (and user
//                     bias) of each upcoming rating into a kDepth-deep shared-memory ring;
//                     P rows of a row group belong to this warp for the whole launch, so the
//                     cursor runs across phase boundaries
//   consume cursor  : the update itself
// Stale-prefetch hazard: the row of rating x is fetched while up to kDepth + 3 earlier ratings are
// still being applied.  The hot loop does not look for it: the packer (pack.cu) marks every rating
// whose user also occurs among the 32 preceding ratings of the stream, and classifies every
// aligned quad, so that the two common cases -- four ratings of one hot item (the item row stays
// in registers: a pure dependent chain, which is what bounds a sub-epoch) and four ratings with
// fresh users and no item repeated back to back -- run as straight-line code; everything else
// takes the generic path, which picks each row's source (registers / prefetch ring / global
// memory) with warp-uniform branches.
// ------------------------------------------------------------------------------------------
template <int E, int KERNEL, int MAXT, bool GATED, bool RING, typename PT = float>
// MAXT: 256 (W <= 8: 255 registers per thread), 384 or 512; GATED: honour update_users /
// update_items (else both on); RING: slabs move between ranks (DSGD), counters and hand-over at
// system scope; PT: storage type of the user-factor rows in HBM (float, __half, __nv_bfloat16)
__global__ void __launch_bounds__(MAXT, 1)
sgd_block_kernel(const SgdParams prm)
{
    constexpr int KPAD = E * 32;
    constexpr unsigned FULL = 0xffffffffu;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int W = prm.W;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int rb = RING ? (int)(blockIdx.x % (unsigned)prm.B) : (int)blockIdx.x;
    // (RING = false: every R.x below is a load from the kernel's parameter bank)
    const SgdRank R = RING ? prm.ranks[blockIdx.x / (unsigned)prm.B] : prm.self;
    __shared__ int abort_s;

    // shared-memory carve-up (every section is a multiple of 16 bytes)
    float *Qs = reinterpret_cast<float *>(smem_raw);
    float *ibs = Qs + (size_t)prm.tile_rows * KPAD;
    PT *prow_all = reinterpret_cast<PT *>(ibs + ((prm.tile_rows + 3) & ~3));
    float *pbias_all = reinterpret_cast<float *>(prow_all + (size_t)W * kDepth * KPAD);
    PackedRating *ring_all = reinterpret_cast<PackedRating *>(pbias_all + (size_t)W * kDepth);
    uint64_t *bars = reinterpret_cast<uint64_t *>(ring_all + (size_t)W * kRing);
    int64_t *boff = reinterpret_cast<int64_t *>(bars + 1 + kStages * W);
    double *se_s = reinterpret_cast<double *>(boff + W * W + 2);
    volatile int32_t *phase_done = reinterpret_cast<volatile int32_t *>(se_s + W);

    PT *prow = prow_all + (size_t)warp * kDepth * KPAD;
    float *pbias = pbias_all + warp * kDepth;
    PackedRating *ring = ring_all + (size_t)warp * kRing;
    uint64_t *tile_bar = bars;
    uint64_t *my_bar = bars + 1 + kStages * warp;

    if (threadIdx.x == 0) {
        mbar_init(tile_bar, 1);
        for (int i = 0; i < kStages * W; ++i) mbar_init(bars + 1 + i, 1);
        for (int i = 0; i < W; ++i) phase_done[i] = 0;
        abort_s = 0;
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }

    const float lr = prm.lr;
    const bool upd_u = !GATED || prm.update_users != 0, upd_i = !GATED || prm.update_items != 0;
    // q' = q + lr (g p - Ki q) = (1 - lr Ki) q + (lr g) p, likewise for p (frozen side: a = 1, gl = 0)
    const float a_i = upd_i ? 1.f - prm.lr * prm.Ki : 1.f;
    const float a_u = upd_u ? 1.f - prm.lr * prm.Ku : 1.f;
    const float a_b = 1.f - prm.lr * prm.Kb;
    const unsigned long long a_i2 = pack2(a_i, a_i), a_u2 = pack2(a_u, a_u);
    const bool upd_bu = (KERNEL == MFREC_KERNEL_LINEAR) || upd_u;
    const bool upd_bi = (KERNEL == MFREC_KERNEL_LINEAR) || upd_i;
    const float fx_scale = prm.fx_scale, fx_inv = prm.fx_inv;
    constexpr uint32_t kRowBytes = KPAD * sizeof(PT);
    PT *const P_rows = reinterpret_cast<PT *>(R.P);
    PT *const P_lane = P_rows + lane * Frag<E>::V;   // this lane's column of every P row
    uint32_t rng = 0x9e3779b9u * (blockIdx.x * 1024u + threadIdx.x + 1u);   // stochastic rounding of bf16 rows
    float *const ub_g = R.ub;
    const int64_t steps_per_epoch = (int64_t)prm.G * prm.B;

    double se = 0.0;          // fp64 total of fp32 per-bucket partials, over the whole launch
    uint32_t chunk_seq = 0;   // chunks this warp has pulled so far (ring stage + mbarrier parity)
    uint32_t tile_seq = 0;    // Q tiles this CTA has pulled so far (mbarrier parity)
    bool chunks_issued = false;   // the first chunks of the coming sub-epoch are already on their way

    // it = (epoch * G + slab step t) * B + sub-epoch s; the slab of a step is (rank + t) mod G.
    // (epoch, t, s) are carried along instead of being decoded from `it`: a 64-bit division per
    // sub-epoch and warp cost 5 % of the epoch.
    int s, t_slab, epoch_rel;
    {
        const int64_t e0 = prm.it_begin / steps_per_epoch;
        const int in0 = (int)(prm.it_begin - e0 * steps_per_epoch);
        epoch_rel = (int)(e0 - prm.e_base);
        t_slab = in0 / prm.B;
        s = in0 - t_slab * prm.B;
    }
    for (int64_t it = prm.it_begin; it < prm.it_end; ++it) {
        const int step = (int)(it - prm.it_begin);
        const int in_epoch = t_slab * prm.B + s;
        int slab = R.rank + t_slab;
        if (slab >= prm.G) slab -= prm.G;
        int cbl = rb + s;
        if (cbl >= prm.B) cbl -= prm.B;
        const int cbg = slab * prm.B + cbl;
        const int cs = R.col_start[cbg * W];
        const int nq = R.col_start[(cbg + 1) * W] - cs;
        // uses of this column block that must be complete before this one: around a ring it is used
        // in every step of every epoch (by one rank after the other), on one device once per epoch
        const int tick_need = RING ? (int)it : epoch_rel * prm.B + s;

        // this CTA's W*W bucket descriptors (worker-major: index w * W + phase) + end sentinel
        const int64_t bucket_base = (((int64_t)slab * prm.B + rb) * prm.B + cbl) * W * W;
        for (int i = threadIdx.x; i <= W * W; i += blockDim.x) boff[i] = R.bucket_off[bucket_base + i];
        // Q tile: one elected thread takes the column block over and issues the bulk copies
        if (threadIdx.x == 0) {
            if (R.ticks) {
                if constexpr (RING) {
                    // the previous user may be another GPU (it pushed the block into this rank's
                    // copy of Q and then released the counter at system scope)
                    const unsigned long long t0 = global_ns();
                    uint32_t polls = 0;
                    while (ld_acquire_sys(R.ticks + cbg) < tick_need) {
                        __nanosleep(128);
                        if ((++polls & 1023u) == 0) {
                            if (*(volatile int32_t *)R.abort) { abort_s = 1; break; }
                            if (prm.wait_ns && global_ns() - t0 > prm.wait_ns) {
                                *(volatile int32_t *)R.abort = 1;
                                abort_s = 1;
                                break;
                            }
                        }
                    }
                } else {
                    while (ld_acquire_gpu(R.ticks + cbg) < tick_need) __nanosleep(64);
                }
                // order the acquire (generic proxy) before the bulk reads (async proxy)
                asm volatile("fence.proxy.async;" ::: "memory");
            }
            bool go = nq > 0;
            if constexpr (RING) go = go && !abort_s;
            if (go) {
                const uint32_t total = (uint32_t)nq * KPAD * 4u;
                mbar_expect_tx(tile_bar, total);
                const char *src = reinterpret_cast<const char *>(R.Q + (size_t)cs * KPAD);
                char *dst = reinterpret_cast<char *>(Qs);
                for (uint32_t o = 0; o < total; o += 32768u)
                    bulk_g2s(dst + o, src + o, min(32768u, total - o), tile_bar);
            }
        }
        __syncthreads();   // descriptors visible; mbarrier init visible (first step)
        if constexpr (RING) {
            if (abort_s) break;   // a hand-over wait timed out (a peer died): leave, the host reports it
        }

        // ---- this warp's stream ---------------------------------------------------------------
        const int64_t S0 = boff[warp * W];
        const uint32_t slen = (uint32_t)(boff[warp * W + W] - S0);   // multiple of 4 (padded buckets)
        const uint32_t nchunks = (slen + kChunk - 1) / kChunk;
        const uint32_t nquads = slen / 4;
        const PackedRating *stream = R.packed + S0;
        const int64_t *off_w = boff + warp * W;

        // Everything below counts in QUADS (4 stream positions = 48 bytes) from the start of this
        // warp's stream: quad x sits in ring slot (base_q + x) mod kRingQ, its P rows in P-ring slots
        // 4 (x mod kQuadsAhead) .., chunk c = quads [16 c, 16 c + 16).
        constexpr uint32_t kRingQ = kRing / 4, kChunkQ = kChunk / 4;
        static_assert((kRingQ & (kRingQ - 1)) == 0 && (kChunkQ & (kChunkQ - 1)) == 0 &&
                      (kQuadsAhead & (kQuadsAhead - 1)) == 0, "ring sizes must be powers of two");
        const uint32_t base_q = (chunk_seq % kStages) * kChunkQ;
        const char *const ring_b = reinterpret_cast<const char *>(ring);
        auto quad_rec = [&](uint32_t x) { return ring_b + ((base_q + x) & (kRingQ - 1)) * 48u; };
        auto chunk_wait = [&](uint32_t c) {
            const uint32_t g = chunk_seq + c;
            mbar_wait(my_bar + (g % kStages), (g / kStages) & 1u);
        };
        auto issue_chunk = [&](uint32_t c) {
            if (lane == 0) {
                const uint32_t cnt = min((uint32_t)kChunk, slen - c * kChunk);
                const uint32_t g = chunk_seq + c;
                uint64_t *bar = my_bar + (g % kStages);
                mbar_expect_tx(bar, cnt * 12u);
                bulk_g2s(ring + (g % kStages) * kChunk, stream + (size_t)c * kChunk, cnt * 12u, bar);
            }
        };
        // (the first chunks of every sub-epoch but the first were requested at the end of the
        // previous one, see below)
        if (!chunks_issued)
            for (uint32_t c = 0; c < nchunks && c < (uint32_t)kStages; ++c) issue_chunk(c);

        // Prefetch: one cp.async group per quad, so group index == quad index.  The first
        // kQuadsAhead - 1 quads are fetched here; after that the rows of quad x + kQuadsAhead - 1
        // are requested WHILE quad x is being applied, one row after each warp reduction, so the
        // copies fill the reduction's latency instead of preceding the dependent chain.  Padding
        // entries name packed user 0, a valid row, and are never consumed.  Quads past the end
        // commit empty groups.
        PT *const prow_lane = prow + lane * Frag<E>::V;
        for (uint32_t fx = 0; fx + 1 < (uint32_t)kQuadsAhead; ++fx) {
            if (fx < nquads) {
                if ((fx & (kChunkQ - 1)) == 0) chunk_wait(fx / kChunkQ);
                const char *rec = quad_rec(fx);
                const uint32_t fslot0 = (fx & (kQuadsAhead - 1)) * 4;
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    const uint32_t ut = *reinterpret_cast<const uint32_t *>(rec + 12 * t) & kIdMask;
                    const PT *gsrc = row_ptr(P_lane, ut, kRowBytes);
#pragma unroll
                    for (int c = 0; c < Frag<E>::NV; ++c)
                        cp_async<Frag<E>::V * sizeof(PT)>(prow_lane + (fslot0 + t) * KPAD + c * 32 * Frag<E>::V,
                                                          gsrc + c * 32 * Frag<E>::V);
                }
                if (lane < 4) {
                    const uint32_t ul = *reinterpret_cast<const uint32_t *>(rec + 12 * lane) & kIdMask;
                    cp_async<4>(pbias + fslot0 + lane, row_ptr(ub_g, ul, 4));
                }
            }
            cp_async_commit();
        }

        if (nq > 0) {
            mbar_wait(tile_bar, tile_seq & 1u);
            tile_seq += 1;
        }
        // item biases of the block: L2 loads (another SM wrote them; L1 may hold a stale line)
        for (int i = threadIdx.x; i < nq; i += blockDim.x) ibs[i] = __ldcg(R.ib + cs + i);
        __syncthreads();   // tile + biases in place

        Frag<E> cp, cq;        // current user row / item row (post-update values)
#pragma unroll
        for (int e = 0; e < E; ++e) { cp.x[e] = 0.f; cq.x[e] = 0.f; }
        float cbu = 0.f, cbi = 0.f, se_f = 0.f;
        int prev_u = -1, prev_i = -1;

        // ---- the arithmetic of one update, on rows held in registers -----------------------------
        // deterministic warp reduction in 32-bit fixed point: one REDUX instead of a 5-level
        // shuffle butterfly; integer addition is associative, so the result does not depend on
        // lane order.  fx_scale is a power of two chosen from max |rating| (see sgd_epoch).
        auto warp_sum_fx = [&](int v) { return __reduce_add_sync(FULL, v); };
        auto dot_fx = [&](const Frag<E> &pu, const Frag<E> &q) {
            float part;
            if constexpr (E >= 2) {
                // two interleaved partial sums (even / odd elements), one packed FMA per pair
                unsigned long long acc = mul2(pack2(pu.x[0], pu.x[1]), pack2(q.x[0], q.x[1]));
#pragma unroll
                for (int e = 2; e < E; e += 2)
                    acc = fma2(pack2(pu.x[e], pu.x[e + 1]), pack2(q.x[e], q.x[e + 1]), acc);
                float lo, hi;
                unpack2(acc, lo, hi);
                part = lo + hi;
            } else {
                part = pu.x[0] * q.x[0];
            }
            return __float2int_rn(part * fx_scale);
        };
        auto apply = [&](int isum, float r, Frag<E> &pu, float &bu, Frag<E> &q, float &bi) {
            const float pred = fmaf((float)isum, fx_inv, bi + bu);
            float err, grad;
            if constexpr (KERNEL == MFREC_KERNEL_LINEAR) {
                err = r - pred;
                grad = err;
            } else {
                const float sig = 1.f / (1.f + expf(-pred));
                err = r - (1.f + 4.f * sig);
                grad = err * sig * (1.f - sig) * 4.f;
            }
            se_f = fmaf(err, err, se_f);
            const float gl = lr * grad;
            bu = upd_bu ? fmaf(a_b, bu, gl) : bu;
            bi = upd_bi ? fmaf(a_b, bi, gl) : bi;
            const float gli = upd_i ? gl : 0.f, glu = upd_u ? gl : 0.f;
            if constexpr (E >= 2) {
                const unsigned long long glu2 = pack2(glu, glu), gli2 = pack2(gli, gli);
#pragma unroll
                for (int e = 0; e < E; e += 2) {
                    const unsigned long long pe = pack2(pu.x[e], pu.x[e + 1]), qe = pack2(q.x[e], q.x[e + 1]);
                    unpack2(fma2(glu2, qe, mul2(a_u2, pe)), pu.x[e], pu.x[e + 1]);
                    unpack2(fma2(gli2, pe, mul2(a_i2, qe)), q.x[e], q.x[e + 1]);
                }
            } else {
                const float pe = pu.x[0], qe = q.x[0];
                pu.x[0] = fmaf(glu, qe, a_u * pe);
                q.x[0] = fmaf(gli, pe, a_i * qe);
            }
        };
        auto store_p_row = [&](int u, const Frag<E> &pu) {
            pfrag_store_lane<E, PT>(pu, row_ptr(P_lane, (uint32_t)u, kRowBytes), rng);
        };
        auto store_p = [&](int u, const Frag<E> &pu, float bu) {
            store_p_row(u, pu);
            if (lane == 0) *row_ptr(ub_g, (uint32_t)u, 4) = bu;
        };
        // the four user biases of a quad in one predicated store: lane t writes rating t's (its
        // user id comes straight from the record).  keep bit t clear = rating t + 1 is the same
        // user and writes the newer value.
        auto store_bias_quad = [&](const int (&u4)[4], const float (&b4)[4], uint32_t keep) {
            const bool lo = (lane & 2) == 0, even = (lane & 1) == 0;
            const int ul = lo ? (even ? u4[0] : u4[1]) : (even ? u4[2] : u4[3]);
            const float v = lo ? (even ? b4[0] : b4[1]) : (even ? b4[2] : b4[3]);
            if (lane < 4 && ((keep >> lane) & 1u)) *row_ptr(ub_g, (uint32_t)ul, 4) = v;
        };
        auto store_q = [&](int it, const Frag<E> &q, float bi) {
            frag_store<E>(q, Qs + (size_t)(it - cs) * KPAD, lane);
            if (lane == 0) ibs[it - cs] = bi;
        };

        // generic path, one rating: sources picked at run time (warp-uniform branches).
        // stale = the packer saw this user among the 32 preceding ratings of the stream, so the
        // prefetched copy of the row may predate an update: take it from registers (adjacent
        // ratings of one user) or re-read it from global memory.
        auto update_one = [&](uint32_t slot, int u, int it, float r, bool stale) {
            Frag<E> pu;
            float bu;
            if (u == prev_u) {
#pragma unroll
                for (int e = 0; e < E; ++e) pu.x[e] = cp.x[e];
                bu = cbu;
            } else if (stale) {
                __syncwarp();   // lane 0's bias store of an earlier rating is visible to every lane
                pfrag_load<E, PT>(pu, row_ptr(P_rows, (uint32_t)u, kRowBytes), lane);
                bu = *row_ptr(ub_g, (uint32_t)u, 4);
            } else {
                pfrag_load<E, PT>(pu, prow + slot * KPAD, lane);
                bu = pbias[slot];
            }
            if (it != prev_i) {   // otherwise the item row is still in registers
                frag_load<E>(cq, Qs + (size_t)(it - cs) * KPAD, lane);
                cbi = ibs[it - cs];
            }
            const int isum = warp_sum_fx(dot_fx(pu, cq));
            apply(isum, r, pu, bu, cq, cbi);
            store_q(it, cq, cbi);
            store_p(u, pu, bu);
#pragma unroll
            for (int e = 0; e < E; ++e) cp.x[e] = pu.x[e];
            cbu = bu;
            prev_u = u;
            prev_i = it;
        };

        // straight-line paths for the quads the packer classified (common.cuh): four fresh,
        // pairwise distinct users, so all four P rows come from the prefetch ring up front
        auto load_quad_p = [&](uint32_t slot0, Frag<E> (&p4)[4], float (&b4)[4]) {
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                pfrag_load<E, PT>(p4[t], prow + (slot0 + t) * KPAD, lane);
                b4[t] = pbias[slot0 + t];
            }
        };
        // kQuadChain: one item; its row stays in registers and is stored once
        auto chain_quad = [&](uint32_t slot0, const int (&u4)[4], int it, const float (&r4)[4], auto &&hook) {
            Frag<E> p4[4];
            float b4[4];
            load_quad_p(slot0, p4, b4);
            if (it != prev_i) {
                frag_load<E>(cq, Qs + (size_t)(it - cs) * KPAD, lane);
                cbi = ibs[it - cs];
            }
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                const int isum = warp_sum_fx(dot_fx(p4[t], cq));
                hook(t);
                apply(isum, r4[t], p4[t], b4[t], cq, cbi);
                store_p_row(u4[t], p4[t]);
            }
            store_bias_quad(u4, b4, 0xfu);
            store_q(it, cq, cbi);
#pragma unroll
            for (int e = 0; e < E; ++e) cp.x[e] = p4[3].x[e];
            cbu = b4[3];
            prev_u = u4[3];
            prev_i = it;
        };
        // kQuadIndep: four ratings that share neither a user nor an item: their order does not
        // matter, so all loads, the four reductions and the four updates are issued side by side
        // (four independent dependency chains for the scheduler instead of one)
        auto indep_quad = [&](uint32_t slot0, const int (&u4)[4], const int (&i4)[4], const float (&r4)[4], auto &&hook) {
            Frag<E> p4[4], q4[4];
            float b4[4], c4[4];
            load_quad_p(slot0, p4, b4);
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                frag_load<E>(q4[t], Qs + (size_t)(i4[t] - cs) * KPAD, lane);
                c4[t] = ibs[i4[t] - cs];
            }
            int f[4], sm[4];
#pragma unroll
            for (int t = 0; t < 4; ++t) f[t] = dot_fx(p4[t], q4[t]);
#pragma unroll
            for (int t = 0; t < 4; ++t) sm[t] = warp_sum_fx(f[t]);
#pragma unroll
            for (int t = 0; t < 4; ++t) hook(t);
#pragma unroll
            for (int t = 0; t < 4; ++t) apply(sm[t], r4[t], p4[t], b4[t], q4[t], c4[t]);
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                store_q(i4[t], q4[t], c4[t]);
                store_p_row(u4[t], p4[t]);
            }
            store_bias_quad(u4, b4, 0xfu);
#pragma unroll
            for (int e = 0; e < E; ++e) { cp.x[e] = p4[3].x[e]; cq.x[e] = q4[3].x[e]; }
            cbu = b4[3];
            cbi = c4[3];
            prev_u = u4[3];
            prev_i = i4[3];
        };
        // kQuadClean: any items; an item row equal to the previous rating's stays in registers
        // (predicated loads, no branch), every updated row goes back to the shared-memory tile
        // (a later rating of the quad may reuse an item: program order through the tile is exact)
        auto clean_quad = [&](uint32_t slot0, const int (&u4)[4], const int (&i4)[4], const int (&f4)[4],
                              const float (&r4)[4], auto &&hook) {
            Frag<E> p4[4];
            float b4[4];
            load_quad_p(slot0, p4, b4);
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                if (f4[t] & kFlagAdjUser) {   // same user as the previous rating: its registers, not the ring
#pragma unroll
                    for (int e = 0; e < E; ++e) p4[t].x[e] = t ? p4[t ? t - 1 : 0].x[e] : cp.x[e];
                    b4[t] = t ? b4[t ? t - 1 : 0] : cbu;
                }
                if (i4[t] != prev_i) {
                    frag_load<E>(cq, Qs + (size_t)(i4[t] - cs) * KPAD, lane);
                    cbi = ibs[i4[t] - cs];
                }
                prev_i = i4[t];
                const int isum = warp_sum_fx(dot_fx(p4[t], cq));
                hook(t);
                apply(isum, r4[t], p4[t], b4[t], cq, cbi);
                store_q(i4[t], cq, cbi);
                store_p_row(u4[t], p4[t]);
            }
            {
                uint32_t keep = 0x8u;
#pragma unroll
                for (int t = 0; t < 3; ++t) keep |= (f4[t + 1] & kFlagAdjUser) ? 0u : (1u << t);
                store_bias_quad(u4, b4, keep);
            }
#pragma unroll
            for (int e = 0; e < E; ++e) cp.x[e] = p4[3].x[e];
            cbu = b4[3];
            prev_u = u4[3];
            prev_i = i4[3];
        };

        const int32_t done_base = step * W;
        uint32_t x = 0;   // quad cursor over the whole stream, runs across the phases
        int4 na = make_int4(0, 0, 0, 0), nb = na, nc = na;   // record of quad x, read ahead
        if (nquads > 0) {   // (its chunk was waited for by the prefetch above)
            const int4 *nsrc = reinterpret_cast<const int4 *>(quad_rec(0));
            na = nsrc[0]; nb = nsrc[1]; nc = nsrc[2];
        }
        for (int p = 0; p < W; ++p) {
            const uint32_t xe = (uint32_t)(off_w[p + 1] - S0) >> 2;   // buckets are padded to quads
            if (p > 0) {
                // column group (warp + p) mod W comes from warp + 1, which used it in phase p - 1
                const volatile int32_t *flag = phase_done + (warp + 1 == W ? 0 : warp + 1);
                if (lane == 0) {
                    while (*flag < done_base + p) __nanosleep(32);
                    __threadfence_block();
                }
                __syncwarp();
            }
            se_f = 0.f;
#pragma unroll 1
            for (; x < xe; ++x) {
                if ((x & (kChunkQ - 1)) == 0 && x != 0) {
                    // entering chunk x / 16: the one before it is consumed, its ring stage is free
                    const uint32_t nc = x / kChunkQ - 1 + kStages;
                    if (nc < nchunks) {
                        __syncwarp();
                        issue_chunk(nc);
                    }
                }
                // the quad whose rows are requested during this iteration; past the end of the
                // stream the last quad's rows are requested again into a free slot (never consumed),
                // which keeps this straight-line code
                const uint32_t fx = x + (kQuadsAhead - 1);
                if ((fx & (kChunkQ - 1)) == 0 && fx < nquads) chunk_wait(fx / kChunkQ);   // first touch of a chunk
                const char *const frec = quad_rec(min(fx, nquads - 1));
                const uint32_t fu[4] = {*reinterpret_cast<const uint32_t *>(frec) & kIdMask,
                                        *reinterpret_cast<const uint32_t *>(frec + 12) & kIdMask,
                                        *reinterpret_cast<const uint32_t *>(frec + 24) & kIdMask,
                                        *reinterpret_cast<const uint32_t *>(frec + 36) & kIdMask};
                const uint32_t fslot0 = (fx & (kQuadsAhead - 1)) * 4;
                PT *const fdst = prow_lane + fslot0 * KPAD;
                auto fetch_row = [&](int t) {
                    const PT *gsrc = row_ptr(P_lane, fu[t], kRowBytes);
#pragma unroll
                    for (int c = 0; c < Frag<E>::NV; ++c)
                        cp_async<Frag<E>::V * sizeof(PT)>(fdst + t * KPAD + c * 32 * Frag<E>::V, gsrc + c * 32 * Frag<E>::V);
                };
                cp_async_wait<kQuadsAhead - 2>();   // the four rows of this quad have landed
                __syncwarp();                       // ... and the bias copies / lane 0's stores are visible
                // this quad's record was read one iteration ago (its decode would otherwise sit in
                // front of everything else with a shared-memory latency); read the next one now
                const int4 a = na, b = nb, c2 = nc;
                {
                    const int4 *nsrc = reinterpret_cast<const int4 *>(quad_rec(x + 1));
                    na = nsrc[0]; nb = nsrc[1]; nc = nsrc[2];
                }
                const uint32_t slot0 = (x & (kQuadsAhead - 1)) * 4;
                const int u4[4] = {a.x & kIdMask, a.w & kIdMask, b.z & kIdMask, c2.y & kIdMask};
                const int f4[4] = {a.y, b.x, b.w, c2.z};   // item ids with the packer's hint bits
                const int i4[4] = {a.y & kIdMask, b.x & kIdMask, b.w & kIdMask, c2.z & kIdMask};
                const float r4[4] = {__int_as_float(a.z), __int_as_float(b.y), __int_as_float(c2.x), __int_as_float(c2.w)};
                const int qtype = (a.x >> kQuadShift) & 3;
                if (qtype == kQuadIndep) {
                    indep_quad(slot0, u4, i4, r4, fetch_row);
                } else if (qtype == kQuadChain) {
                    chain_quad(slot0, u4, i4[0], r4, fetch_row);
                } else if (qtype == kQuadClean) {
                    clean_quad(slot0, u4, i4, f4, r4, fetch_row);
                } else {
#pragma unroll
                    for (int t = 0; t < 4; ++t) {
                        if (!(f4[t] & kFlagPad)) update_one(slot0 + t, u4[t], i4[t], r4[t], (f4[t] & kFlagStale) != 0);
                        fetch_row(t);
                    }
                }
                {
                    // lane t < 4 requests the bias of row t; ids picked from registers (a load from
                    // the record here would put its latency at the end of every iteration)
                    const bool lo = (lane & 2) == 0, even = (lane & 1) == 0;
                    const uint32_t ul = lo ? (even ? fu[0] : fu[1]) : (even ? fu[2] : fu[3]);
                    if (lane < 4) cp_async<4>(pbias + fslot0 + lane, row_ptr(ub_g, ul, 4));
                }
                cp_async_commit();
            }
            se += (double)se_f;
            prev_i = -1;       // the column group changes hands: never forward Q across a phase
            // hand the column group over: Q rows / item biases written above, then the counter
            __syncwarp();
            if (lane == 0) {
                __threadfence_block();
                phase_done[warp] = done_base + p + 1;
            }
        }
        cp_async_wait<0>();
        chunk_seq += nchunks;
        // This warp's rating ring is free: request the first chunks of its next sub-epoch's stream
        // now, so that they cross while the CTA waits for its last warp, writes the tile back and
        // waits for the next column block (the stream does not depend on any other CTA).
        chunks_issued = false;
        // (s, t) of the next iteration
        int ns = s + 1, nt = t_slab;
        if (ns == prm.B) {
            ns = 0;
            nt = t_slab + 1 == prm.G ? 0 : t_slab + 1;
        }
        if (it + 1 < prm.it_end) {
            int nslab = R.rank + nt;
            if (nslab >= prm.G) nslab -= prm.G;
            int ncbl = rb + ns;
            if (ncbl >= prm.B) ncbl -= prm.B;
            const int64_t nbase = ((((int64_t)nslab * prm.B + rb) * prm.B + ncbl) * W + warp) * W;
            const int64_t nS0 = __ldg(R.bucket_off + nbase);
            const uint32_t nslen = (uint32_t)(__ldg(R.bucket_off + nbase + W) - nS0);
            const uint32_t nn = min((nslen + kChunk - 1) / kChunk, (uint32_t)kStages);
            if (lane == 0) {
                for (uint32_t c = 0; c < nn; ++c) {
                    const uint32_t cnt = min((uint32_t)kChunk, nslen - c * kChunk);
                    const uint32_t g = chunk_seq + c;
                    uint64_t *bar = my_bar + (g % kStages);
                    mbar_expect_tx(bar, cnt * 12u);
                    bulk_g2s(ring + (g % kStages) * kChunk, R.packed + nS0 + (size_t)c * kChunk, cnt * 12u, bar);
                }
            }
            chunks_issued = true;
        }
        __syncthreads();   // every warp is done with the tile
        // write the Q tile back and pass the column block on.  Around a ring the last sub-epoch of
        // a step leaves the block in the NEXT rank's copy of Q (peer memory, over NVLink): that
        // rank finds it in its own HBM when the counter arrives.
        const bool to_peer = RING && s + 1 == prm.B && prm.world > 1;
        {
            const int nvec = nq * KPAD / 4;
            float4 *dst = reinterpret_cast<float4 *>((to_peer ? R.peer_Q : R.Q) + (size_t)cs * KPAD);
            float *dst_b = (to_peer ? R.peer_ib : R.ib) + cs;
            const float4 *srcv = reinterpret_cast<const float4 *>(Qs);
            // Divergence check, off the hot loop: the fixed-point reduction turns a NaN partial
            // into 0, so a non-finite factor would never reach the error sum -- but any update
            // with a non-finite P or Q row leaves a non-finite Q row, and every Q row passes
            // through here.  0 * x is NaN exactly for x = +-inf / NaN.
            float chk = 0.f;
            for (int i = threadIdx.x; i < nvec; i += blockDim.x) {
                const float4 t = srcv[i];
                chk = fmaf(0.f, t.x, fmaf(0.f, t.y, fmaf(0.f, t.z, fmaf(0.f, t.w, chk))));
                dst[i] = t;
            }
            for (int i = threadIdx.x; i < nq; i += blockDim.x) {
                chk = fmaf(0.f, ibs[i], chk);
                dst_b[i] = ibs[i];
            }
            if (__any_sync(FULL, chk != chk)) se = NAN;   // the reference prints a NaN RMSE then (kmf_train.pyx:273)
        }
        // the epoch's error sum leaves with its last sub-epoch (or with the launch)
        const bool epoch_ends = in_epoch + 1 == (int)steps_per_epoch || it + 1 == prm.it_end;
        if (epoch_ends) {
            if (lane == 0) se_s[warp] = se;
            se = 0.0;
        }
        if (R.ticks) {
            if constexpr (RING) {
                if (to_peer) {
                    __threadfence_system();
                    __syncthreads();
                    if (threadIdx.x == 0) st_release_sys(R.peer_ticks + cbg, tick_need + 1);
                } else {
                    // last sub-epoch of a step on a single rank (world == 1 never takes RING) or
                    // an inner sub-epoch: the next user is a CTA of this device
                    __threadfence();
                    __syncthreads();
                    if (threadIdx.x == 0) st_release_gpu(R.ticks + cbg, tick_need + 1);
                }
            } else {
                __threadfence();
                __syncthreads();
                if (threadIdx.x == 0) st_release_gpu(R.ticks + cbg, tick_need + 1);
            }
        } else {
            __syncthreads();
        }
        if (epoch_ends && threadIdx.x == 0) {
            double tot = 0.0;
            for (int w = 0; w < W; ++w) tot += se_s[w];
            R.se_part[(int64_t)epoch_rel * prm.se_stride + rb] = tot;
        }
        if (ns == 0 && nt == 0) epoch_rel += 1;
        s = ns;
        t_slab = nt;
    }
    if constexpr (RING) {
        // timed out: every epoch this launch still owed reports NaN
        if (abort_s && threadIdx.x == 0) {
            const int64_t e_last = (prm.it_end - 1) / steps_per_epoch;
            for (int64_t e = prm.e_base; e <= e_last; ++e) R.se_part[(e - prm.e_base) * prm.se_stride + rb] = NAN;
        }
    }
}

// fixed-order sum of the per-CTA partials of one epoch
__global__ void __launch_bounds__(1024) se_reduce_kernel(const double *__restrict__ part, int64_t n,
                                                         double *__restrict__ out)
{
    __shared__ double sh[1024];
    double acc = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += 1024) acc += part[i];
    sh[threadIdx.x] = acc;
    __syncthreads();
    for (int o = 512; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) *out = sh[0];
}

// Hot-item copies (pack.cu): after an epoch every split item's copies are replaced by their mean,
// rows and biases alike.  One warp per item, fixed summation order: deterministic.  Around a ring
// the rank that holds the slab merges it, after its neighbour's last pushes have arrived
// (ticks != null: wait until counters [tick_lo, tick_hi) reach tick_need, system scope).
__global__ void __launch_bounds__(256)
merge_copies_kernel(float *__restrict__ Q, float *__restrict__ ib, int kpad, const int32_t *__restrict__ hot_off,
                    const int32_t *__restrict__ hot_rows, int32_t n_hot, int32_t row_lo, int32_t row_hi,
                    const int32_t *ticks, int32_t tick_lo, int32_t tick_hi, int32_t tick_need,
                    int32_t *abort_flag, unsigned long long wait_ns)
{
    __shared__ int ok;
    if (ticks) {
        if (threadIdx.x == 0) {
            ok = 1;
            const unsigned long long t0 = global_ns();
            for (int32_t c = tick_lo; c < tick_hi && ok; ++c) {
                uint32_t polls = 0;
                while (ld_acquire_sys(ticks + c) < tick_need) {
                    __nanosleep(256);
                    if ((++polls & 255u) == 0 &&
                        (*(volatile int32_t *)abort_flag || (wait_ns && global_ns() - t0 > wait_ns))) {
                        *(volatile int32_t *)abort_flag = 1;
                        ok = 0;
                        break;
                    }
                }
            }
        }
        __syncthreads();
        if (!ok) return;
    }
    const int lane = threadIdx.x & 31;
    const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t h = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; h < n_hot; h += warps) {
        const int32_t a = hot_off[h], b = hot_off[h + 1];
        const int32_t first = hot_rows[a];
        if (first < row_lo || first >= row_hi) continue;   // (all copies of an item live in one slab)
        const float inv = 1.f / (float)(b - a);
        for (int c = lane; c < kpad; c += 32) {
            float acc = 0.f;
            for (int32_t j = a; j < b; ++j) acc += __ldcg(Q + (size_t)hot_rows[j] * kpad + c);
            acc *= inv;
            for (int32_t j = a; j < b; ++j) Q[(size_t)hot_rows[j] * kpad + c] = acc;
        }
        if (lane == 0) {
            float acc = 0.f;
            for (int32_t j = a; j < b; ++j) acc += __ldcg(ib + hot_rows[j]);
            acc *= inv;
            for (int32_t j = a; j < b; ++j) ib[hot_rows[j]] = acc;
        }
    }
}

// ------------------------------------------------------------------------------------------
// Sequential schedule: the reference's loop (kmf_train.pyx:241-273) in the reference's ORDER,
// fp64, round-to-nearest multiplies and adds kept separate (the reference build has no FMA).
//
// One warp takes the rating stream 32 ratings at a time, one rating per lane.  Two ratings only
// interact through the rows / biases of a shared user or item, so the lanes compute the
// dependency level of their rating inside the window (1 + the level of the latest earlier rating
// with the same user / the same item) and the window runs level by level: the lanes of a level
// touch disjoint rows, levels run in order, every lane's own arithmetic (the dot product summed
// over f in order, the update) is the reference's -- the result is bit-identical to one thread
// walking the stream, in (levels) steps per window instead of 32.  Shuffled ratings rarely share
// a user or an item within 32 consecutive entries: almost every window is a single level.  The
// squared errors are summed in stream order (the printed RMSE is the reference's, too).
// ------------------------------------------------------------------------------------------
constexpr int kSeqRegs = 32;   // features of a row pair kept in registers by the sequential kernel

// A float64 factor row: feature f at p[f * stride].  RO rows are read through the read-only path
// and never written (the frozen side of a batched fold-in).
template <bool RO>
struct KmfRow {
    double *p;
    int64_t stride;
    __device__ __forceinline__ double ld(int f) const
    {
        if constexpr (RO) return __ldg(p + (int64_t)f * stride);
        else return p[(int64_t)f * stride];
    }
    __device__ __forceinline__ void st(int f, double x) const
    {
        if constexpr (!RO) p[(int64_t)f * stride] = x;
    }
};

// One rating of the reference loop (kmf_train.pyx:241-273 linear, :150-185 logistic): the prediction
// summed over f in order, the error, the bias updates, then the feature updates -- every multiply and
// add rounded on its own.  Every schedule that must reproduce the reference calls this one function,
// so their results agree by construction.  bi / bu: the item / user bias (a register or the array
// element itself), replaced by its updated value where the reference updates it (the linear kernel
// updates both unconditionally).
// Returns the squared error.
template <class IRow, class URow>
__device__ __forceinline__ double kmf_rating(int kernel, int dim, double lr, double K_users, double K_items,
                                             double K_bias, double r, const IRow &ui_, const URow &vu_,
                                             double &bi, double &bu, int update_users, int update_items)
{
    const double bi0 = bi, bu0 = bu;
    double s = __dadd_rn(__dadd_rn(0.0, bi0), bu0);
    double e2 = 0.0;
    auto err_grad = [&](double &err, double &grad) {
        if (kernel == MFREC_KERNEL_LINEAR) {
            err = __dadd_rn(r, -s);
            grad = err;
        } else {
            const double sig = 1.0 / __dadd_rn(1.0, exp(-s));
            const double p = __dadd_rn(1.0, __dmul_rn(sig, 4.0));
            err = __dadd_rn(r, -p);
            grad = __dmul_rn(__dmul_rn(__dmul_rn(err, sig), __dadd_rn(1.0, -sig)), 4.0);
        }
        e2 = __dmul_rn(err, err);
        if (kernel == MFREC_KERNEL_LINEAR || update_users)
            bu = __dadd_rn(bu0, __dmul_rn(lr, __dadd_rn(grad, -__dmul_rn(K_bias, bu0))));
        if (kernel == MFREC_KERNEL_LINEAR || update_items)
            bi = __dadd_rn(bi0, __dmul_rn(lr, __dadd_rn(grad, -__dmul_rn(K_bias, bi0))));
    };
    double err, grad;
    if (dim <= kSeqRegs) {
        // both rows fit in registers: every load of the rating is in flight at once, the
        // sum runs over f in order, the update reuses the registers
        double mf[kSeqRegs], cf[kSeqRegs];
#pragma unroll
        for (int f = 0; f < kSeqRegs; ++f)
            if (f < dim) { mf[f] = ui_.ld(f); cf[f] = vu_.ld(f); }
#pragma unroll
        for (int f = 0; f < kSeqRegs; ++f)
            if (f < dim) s = __dadd_rn(s, __dmul_rn(mf[f], cf[f]));
        err_grad(err, grad);
#pragma unroll
        for (int f = 0; f < kSeqRegs; ++f) {
            if (f >= dim) continue;
            if (update_items)
                ui_.st(f, __dadd_rn(mf[f], __dmul_rn(lr, __dadd_rn(__dmul_rn(grad, cf[f]), -__dmul_rn(K_items, mf[f])))));
            if (update_users)
                vu_.st(f, __dadd_rn(cf[f], __dmul_rn(lr, __dadd_rn(__dmul_rn(grad, mf[f]), -__dmul_rn(K_users, cf[f])))));
        }
    } else {
        // rows are read eight features at a time (independent loads in flight together)
        for (int f0 = 0; f0 < dim; f0 += 8) {
            double a[8], b[8];
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if (f0 + j < dim) { a[j] = ui_.ld(f0 + j); b[j] = vu_.ld(f0 + j); }
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if (f0 + j < dim) s = __dadd_rn(s, __dmul_rn(a[j], b[j]));
        }
        err_grad(err, grad);
        for (int f0 = 0; f0 < dim; f0 += 8) {
            double mf[8], cf[8];
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if (f0 + j < dim) { mf[j] = ui_.ld(f0 + j); cf[j] = vu_.ld(f0 + j); }
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                if (f0 + j >= dim) continue;
                if (update_items)
                    ui_.st(f0 + j, __dadd_rn(mf[j], __dmul_rn(lr, __dadd_rn(__dmul_rn(grad, cf[j]), -__dmul_rn(K_items, mf[j])))));
                if (update_users)
                    vu_.st(f0 + j, __dadd_rn(cf[j], __dmul_rn(lr, __dadd_rn(__dmul_rn(grad, mf[j]), -__dmul_rn(K_users, cf[j])))));
            }
        }
    }
    return e2;
}

__global__ void __launch_bounds__(32)
kmf_sequential_kernel(int kernel, int nbr_epochs, int dim, double lr, double K_users,
                      double K_items, double K_bias, double *u, double *v,
                      const int32_t *idx, const double *ratings, int64_t nnz,
                      int64_t ni, int64_t nu, double *ib, double *ub,
                      int update_users, int update_items, double *rmse_out)
{
    if (blockIdx.x != 0) return;
    const int lane = threadIdx.x;
    const unsigned FULLM = 0xffffffffu;
    for (int epoch = 0; epoch < nbr_epochs; ++epoch) {
        double se = 0.0;
        int2 ui = make_int2(0, 0);
        double rating = 0.0;
        if (lane < nnz) { ui = reinterpret_cast<const int2 *>(idx)[lane]; rating = ratings[lane]; }
        for (int64_t base = 0; base < nnz; base += 32) {
            const int cnt = (int)(nnz - base < 32 ? nnz - base : 32);
            const bool live = lane < cnt;
            const int user = ui.x, item = ui.y;
            const double r = rating;
            {   // the next window's ratings, in flight while this one runs
                const int64_t j = base + 32 + lane;
                if (j < nnz) { ui = reinterpret_cast<const int2 *>(idx)[j]; rating = ratings[j]; }
            }
            int lmax;
            const int level = mfrec_window_levels(user, item, live, lane, lmax);   // common.cuh
            double e2 = 0.0;
            for (int L = 1; L <= lmax; ++L) {
                if (live && level == L) {
                    e2 = kmf_rating(kernel, dim, lr, K_users, K_items, K_bias, r, KmfRow<false>{u + item, ni},
                                    KmfRow<false>{v + user, nu}, ib[item], ub[user], update_users, update_items);
                }
                __syncwarp();   // this level's stores are visible to the lanes of the next
            }
            for (int t = 0; t < cnt; ++t) se = __dadd_rn(se, __shfl_sync(FULLM, e2, t));   // stream order
        }
        if (rmse_out && lane == 0) rmse_out[epoch] = sqrt(se / (double)nnz);
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------
// Batched fold-in (mfrec_fold_in_kmf): many fold-ins of the kind KMFRecommender.retrain_user /
// retrain_item / add_user make (kmf.py:120-172), each ONE row trained on its own ratings against a
// frozen other side.  All ratings of a fold-in share that row, so a fold-in is one serial chain:
// ONE LANE PER ROW.  The lane walks its row's ratings in input order nbr_epochs times through
// kmf_rating, the arithmetic of kmf_sequential_kernel, and sums the squared errors in the same
// order: the result is the per-row call's bit for bit.
//
// The trained row stays on chip in a per-lane slice of shared memory, lane-interleaved (feature f of
// lane t at slice[f * lanes + t]: no bank conflicts); only when not even one lane's row fits in
// shared memory (k > ~29k) does it stay in its global row.  The frozen rows ([m][k], one contiguous
// row per rating) go through the read-only path.  Jobs = rows with at least one rating, in launch
// order; job j's ratings are [job_ptr[j], job_ptr[j+1]), its row is job_row[j] of trained / tbias.
// Jobs of one launch share no written state: with the logistic kernel nothing of the frozen side
// is written, with the linear kernel its biases are (the reference updates them unconditionally),
// so the host launches one level of rows at a time (mfrec_fold_in_kmf).
// ------------------------------------------------------------------------------------------
template <bool SMEM, int SIDE>
__global__ void __launch_bounds__(32)
kmf_fold_in_kernel(int kernel, int nbr_epochs, int dim, double lr, double K_users, double K_items,
                   double K_bias, double *__restrict__ trained, double *__restrict__ tbias,
                   const double *__restrict__ frozen, double *fbias, const int32_t *__restrict__ job_row,
                   const int64_t *__restrict__ job_ptr, const int32_t *__restrict__ fidx,
                   const double *__restrict__ rv, int32_t n_jobs, double *__restrict__ rmse)
{
    extern __shared__ double slice[];
    const int lanes = blockDim.x, t = threadIdx.x;
    const int32_t j = blockIdx.x * lanes + t;
    if (j >= n_jobs) return;
    const int32_t row = job_row[j];
    double *const grow = trained + (size_t)row * dim;
    const KmfRow<false> mine{SMEM ? slice + t : grow, SMEM ? lanes : 1};
    if (SMEM)
        for (int f = 0; f < dim; ++f) mine.st(f, grow[f]);
    double b = tbias[row];
    const int64_t a = job_ptr[j], e = job_ptr[j + 1];
    const bool linear = kernel == MFREC_KERNEL_LINEAR;
    for (int epoch = 0; epoch < nbr_epochs; ++epoch) {
        double se = 0.0;
        for (int64_t n = a; n < e; ++n) {
            const int32_t c = fidx[n];
            const double r = rv[n];
            const KmfRow<true> other{const_cast<double *>(frozen) + (size_t)c * dim, 1};
            double fb = linear ? fbias[c] : __ldg(fbias + c);
            const double e2 = SIDE == MFREC_FOLD_USERS
                ? kmf_rating(kernel, dim, lr, K_users, K_items, K_bias, r, other, mine, fb, b, 1, 0)
                : kmf_rating(kernel, dim, lr, K_users, K_items, K_bias, r, mine, other, b, fb, 0, 1);
            if (linear) fbias[c] = fb;
            se = __dadd_rn(se, e2);
        }
        rmse[(size_t)j * nbr_epochs + epoch] = sqrt(se / (double)(e - a));
    }
    if (SMEM)
        for (int f = 0; f < dim; ++f) grow[f] = mine.ld(f);
    tbias[row] = b;
}

}  // namespace

// shared memory one CTA of the stratified kernel needs (also used by pack.cu to size blocks)
size_t mfrec_sgd_smem_bytes(int tile_rows, int kpad, int W, int p_elem_bytes)
{
    size_t b = (size_t)tile_rows * kpad * 4;               // Q tile
    b += (size_t)((tile_rows + 3) & ~3) * 4;               // item biases
    b += (size_t)W * kDepth * kpad * p_elem_bytes;         // P-row rings (in the rows' storage type)
    b += (size_t)W * kDepth * 4;                           // user-bias rings
    b += (size_t)W * kRing * sizeof(PackedRating);         // rating rings
    b += (size_t)(1 + kStages * W) * 8;                    // mbarriers
    b += (size_t)(W * W + 2) * 8;                          // bucket offsets (padded quads make counts redundant)
    b += (size_t)W * 8;                                    // per-warp squared error
    b += (size_t)((W + 3) & ~3) * 4;                       // per-warp phase counters
    return b + 384;   // alignment of the dynamic window + the kernel's static shared variables
}

namespace {

template <int E>
int launch_sgd(mfrec_ctx *ctx, int kernel, SgdParams &prm, size_t smem, bool cooperative, int grid, bool ring,
               int p_kind)
{
    const bool wide = prm.W > 8;
    // both sides updated (the training call) gets the variant without the gates; fold-in calls
    // (update_users / update_items = 0) the gated one
    const bool gated = !(prm.update_users && prm.update_items);
    void (*fn)(const SgdParams) = nullptr;
    // 9..12 warps: 384 threads leave 170 registers per thread (the kernel needs ~165: no spills);
    // 13..16 warps run the 512-thread build (128 registers, spills)
    const bool mid = prm.W > 8 && prm.W <= 12 && !gated;
#define MF_PICK(K)                                                                                     \
    fn = mid ? sgd_block_kernel<E, K, 384, false, false>                                                \
       : wide ? (gated ? sgd_block_kernel<E, K, 512, true, false> : sgd_block_kernel<E, K, 512, false, false>) \
              : (gated ? sgd_block_kernel<E, K, 256, true, false> : sgd_block_kernel<E, K, 256, false, false>)
#define MF_PICK_RING(K) \
    fn = mid ? sgd_block_kernel<E, K, 384, false, true>                                                  \
       : wide ? sgd_block_kernel<E, K, 512, false, true> : sgd_block_kernel<E, K, 256, false, true>
    if (p_kind != MFREC_STORAGE_F32) {
        // 16-bit user-factor rows: the training build only (both sides updated, <= 12 warps, one device)
        if constexpr (E >= 2) {
            if (ring || gated || prm.W > 12)
                return mfrec_set_error(ctx, MFREC_ERR_UNSUPPORTED,
                                       "fp16 / bf16 user-factor storage: single device, both sides updated, at most 12 warps per CTA");
#define MF_PICK16(K, T) fn = prm.W > 8 ? sgd_block_kernel<E, K, 384, false, false, T> : sgd_block_kernel<E, K, 256, false, false, T>
            if (kernel == MFREC_KERNEL_LINEAR) {
                if (p_kind == MFREC_STORAGE_F16) { MF_PICK16(MFREC_KERNEL_LINEAR, __half); } else { MF_PICK16(MFREC_KERNEL_LINEAR, __nv_bfloat16); }
            } else {
                if (p_kind == MFREC_STORAGE_F16) { MF_PICK16(MFREC_KERNEL_LOGISTIC, __half); } else { MF_PICK16(MFREC_KERNEL_LOGISTIC, __nv_bfloat16); }
            }
#undef MF_PICK16
        } else {
            return mfrec_set_error(ctx, MFREC_ERR_UNSUPPORTED, "fp16 / bf16 user-factor storage needs k > 32");
        }
    } else if (ring) {
        if (gated)
            return mfrec_set_error(ctx, MFREC_ERR_UNSUPPORTED, "ring launches train both sides");
        if (kernel == MFREC_KERNEL_LINEAR) { MF_PICK_RING(MFREC_KERNEL_LINEAR); } else { MF_PICK_RING(MFREC_KERNEL_LOGISTIC); }
    } else {
        if (kernel == MFREC_KERNEL_LINEAR) { MF_PICK(MFREC_KERNEL_LINEAR); } else { MF_PICK(MFREC_KERNEL_LOGISTIC); }
    }
#undef MF_PICK
#undef MF_PICK_RING
    // per device and cheap: set on every launch (a process may hold contexts on several devices)
    MF_CUDA(ctx, cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (cooperative) {
        // all CTAs must be resident at once: they wait on one another's column blocks
        void *args[] = {(void *)&prm};
        MF_CUDA(ctx, cudaLaunchCooperativeKernel((const void *)fn, dim3(grid), dim3(prm.W * 32), args, smem,
                                                 ctx->stream));
        ctx->launches += 1;
    } else {
        fn<<<grid, prm.W * 32, smem, ctx->stream>>>(prm);
        MF_LAUNCH_CHECK(ctx);
    }
    return MFREC_OK;
}

int launch_sgd_kpad(mfrec_ctx *ctx, int kpad, int kernel, SgdParams &prm, size_t smem, bool cooperative,
                    int grid = 0, bool ring = false, int p_kind = MFREC_STORAGE_F32)
{
    if (grid == 0) grid = prm.B;
    switch (kpad) {
    case 32: return launch_sgd<1>(ctx, kernel, prm, smem, cooperative, grid, ring, p_kind);
    case 64: return launch_sgd<2>(ctx, kernel, prm, smem, cooperative, grid, ring, p_kind);
    case 128: return launch_sgd<4>(ctx, kernel, prm, smem, cooperative, grid, ring, p_kind);
    case 256: return launch_sgd<8>(ctx, kernel, prm, smem, cooperative, grid, ring, p_kind);
    default: return mfrec_set_error(ctx, MFREC_ERR_UNSUPPORTED, "kpad=%d", kpad);
    }
}

// can n CTAs of W warps with `smem` bytes each be co-resident (one wave)?
bool sgd_fits_one_wave(mfrec_ctx *ctx, int n, int W, size_t smem)
{
    // one CTA per SM is always possible when the shared memory fits (<= 512 threads, <= 128
    // registers per thread by __launch_bounds__); more than sm_count CTAs would need two per SM
    if (n <= ctx->sm_count) return smem <= ctx->smem_optin;
    const size_t per_sm = ctx->smem_per_sm;
    const int by_smem = (int)(per_sm / (smem + 1024));
    const int by_threads = 2048 / (W * 32);
    const int by_regs = 65536 / (128 * W * 32);
    const int per = std::min(by_smem, std::min(by_threads, by_regs));
    return (int64_t)per * ctx->sm_count >= n;
}

// hyper-parameters + the fixed-point scale of the warp reduction
void fill_hyper(SgdParams &prm, const mfrec_ratings *r, double learning_rate, double K_users, double K_items,
                double K_bias, int update_users, int update_items)
{
    prm.lr = (float)learning_rate; prm.Ku = (float)K_users; prm.Ki = (float)K_items; prm.Kb = (float)K_bias;
    prm.update_users = update_users; prm.update_items = update_items;
    // The dot product's cross-lane sum runs in 32-bit fixed point (REDUX).  Predictions live
    // on the rating scale, so allow |dot| up to 16 x max|rating| (at least 16) before the
    // integer sum wraps; the resolution is then <= 2^-23 of that range (fp32-like).  A run that
    // diverges leaves that range on its way to inf / NaN factors, which the kernel reports as a
    // NaN error sum (see the tile write-back in sgd_block_kernel).
    const float range = 16.f * fmaxf(r->max_abs_rating, 1.f);
    int ex = 0;
    frexpf(range, &ex);              // range <= 2^ex
    prm.fx_scale = ldexpf(1.f, 30 - ex);
    prm.fx_inv = ldexpf(1.f, ex - 30);
    prm.wait_ns = 0;
    prm.ranks = nullptr;
}

int ensure_scratch(mfrec_ctx *ctx, size_t se_doubles, size_t ticks)
{
    if (ctx->se_cap < se_doubles) {
        if (ctx->se_scratch) cudaFree(ctx->se_scratch);
        ctx->se_scratch = nullptr;
        ctx->se_cap = 0;
        MF_CUDA(ctx, cudaMalloc((void **)&ctx->se_scratch, se_doubles * 8));
        ctx->se_cap = se_doubles;
    }
    if (ctx->ticks_cap < ticks) {
        if (ctx->ticks) cudaFree(ctx->ticks);
        ctx->ticks = nullptr;
        ctx->ticks_cap = 0;
        MF_CUDA(ctx, cudaMalloc((void **)&ctx->ticks, ticks * 4));
        ctx->ticks_cap = ticks;
    }
    return MFREC_OK;
}

}  // namespace

int mfrec_merge_copies(mfrec_ctx *ctx, float *Q, float *ib, int kpad, const int32_t *hot_off,
                       const int32_t *hot_rows, int32_t n_hot, int32_t row_lo, int32_t row_hi,
                       const int32_t *ticks, int32_t tick_lo, int32_t tick_hi, int32_t tick_need,
                       int32_t *abort_flag, unsigned long long wait_ns)
{
    if (n_hot <= 0) return MFREC_OK;
    const int blocks = std::max(1, std::min((n_hot + 7) / 8, ctx->sm_count));
    merge_copies_kernel<<<blocks, 256, 0, ctx->stream>>>(Q, ib, kpad, hot_off, hot_rows, n_hot, row_lo, row_hi, ticks,
                                                         tick_lo, tick_hi, tick_need, abort_flag, wait_ns);
    MF_LAUNCH_CHECK(ctx);
    return MFREC_OK;
}

extern "C" int mfrec_sgd_epoch(mfrec_ctx *ctx, const mfrec_ratings *r, mfrec_model *m, int kernel,
                               double learning_rate, double K_users, double K_items, double K_bias,
                               int update_users, int update_items, int32_t slab, double *sq_err_out)
{
    if (!ctx || !r || !m) return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_sgd_epoch: NULL argument");
    if (kernel != MFREC_KERNEL_LINEAR && kernel != MFREC_KERNEL_LOGISTIC)
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_sgd_epoch: kernel=%d", kernel);
    if (m->ni != r->ni || m->nu != r->nu || !m->user_perm || m->ni_rows != r->ni_v)
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_sgd_epoch: model was not created with this layout");
    if (slab >= r->G) return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_sgd_epoch: slab=%d of %d", slab, r->G);
    if (slab >= 0 && r->n_hot > 0)
        return mfrec_set_error(ctx, MFREC_ERR_UNSUPPORTED,
                               "mfrec_sgd_epoch: a layout with hot-item copies is trained a whole epoch at a time (its copies are "
                               "merged at the end of the epoch); pack with opts.split = MFREC_SPLIT_OFF to drive single slabs");
    MF_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t smem = mfrec_sgd_smem_bytes(r->max_cb_items, m->kpad, r->W, m->p_kind == MFREC_STORAGE_F32 ? 4 : 2);
    if (smem > ctx->smem_optin)
        return mfrec_set_error(ctx, MFREC_ERR_UNSUPPORTED,
                               "mfrec_sgd_epoch: Q tile of %d rows x %d needs %zu B shared memory (> %zu); pack with more row_blocks",
                               r->max_cb_items, m->kpad, smem, ctx->smem_optin);
    // MFREC_SGD_LAUNCH_PER_SUBEPOCH=1 forces the fallback (one launch per sub-epoch, no hand-over)
    static int per_subepoch_env = -1;
    if (per_subepoch_env < 0) per_subepoch_env = getenv("MFREC_SGD_LAUNCH_PER_SUBEPOCH") ? 1 : 0;
    const bool persistent = !per_subepoch_env && ctx->coop_launch && sgd_fits_one_wave(ctx, r->B, r->W, smem);
    // The flattened iteration space of the kernel: it = (epoch * G + step) * B + s with the slab of
    // a step = (rank + step) mod G.  The whole epoch = steps 0 .. G-1 as rank 0; one slab = step 0
    // as "rank" slab.
    const int rank = slab < 0 ? 0 : slab;
    const int64_t n_it = (int64_t)(slab < 0 ? r->G : 1) * r->B;
    const int64_t launches = persistent ? 1 : n_it;
    const int64_t nparts = launches * r->B;
    MF_TRY(ensure_scratch(ctx, (size_t)nparts, persistent ? (size_t)r->G * r->B : 0));
    SgdParams prm;
    memset(&prm, 0, sizeof(prm));
    fill_hyper(prm, r, learning_rate, K_users, K_items, K_bias, update_users, update_items);
    prm.self.packed = r->packed;
    prm.self.bucket_off = r->bucket_off;
    prm.self.col_start = r->col_start;
    prm.self.Q = m->Q; prm.self.ib = m->ib; prm.self.P = m->P; prm.self.ub = m->ub;
    prm.self.rank = rank;
    prm.B = r->B; prm.W = r->W; prm.G = r->G; prm.world = 1;
    prm.tile_rows = r->max_cb_items;
    prm.e_base = 0;
    prm.se_stride = r->B;
    int64_t part = 0;
    for (int64_t it = 0; it < n_it; it += persistent ? n_it : 1) {
        prm.it_begin = it;
        prm.it_end = persistent ? n_it : it + 1;
        prm.self.ticks = persistent ? ctx->ticks : nullptr;
        prm.self.se_part = ctx->se_scratch + part;
        part += r->B;
        if (persistent) MF_CUDA(ctx, cudaMemsetAsync(ctx->ticks, 0, (size_t)r->G * r->B * 4, ctx->stream));
        MF_TRY(launch_sgd_kpad(ctx, m->kpad, kernel, prm, smem, persistent, 0, false, m->p_kind));
    }
    if (sq_err_out) {
        se_reduce_kernel<<<1, 1024, 0, ctx->stream>>>(ctx->se_scratch, nparts, sq_err_out);
        MF_LAUNCH_CHECK(ctx);
    }
    // the epoch is complete: merge the copies of the split items
    MF_TRY(mfrec_merge_copies(ctx, m->Q, m->ib, m->kpad, m->hot_off, m->hot_rows, m->n_hot, 0, m->ni_rows, nullptr, 0, 0, 0,
                              nullptr, 0));
    return MFREC_OK;
}

// ------------------------------------------------------------------------------------------
// DSGD ring (SURVEY.md 8(e)): `world` ranks = `world` user slices x `world` item slabs.  Rank r
// keeps its users' P rows and ratings; in step t of an epoch it updates its users x slab
// (r + t) mod world.  ONE persistent launch per rank covers any number of epochs: a column block
// is handed from CTA to CTA inside the device exactly as on one GPU, and the LAST sub-epoch of a
// step writes the block straight into the NEXT rank's copy of Q (peer memory over NVLink:
// cudaIpc-mapped across processes, directly addressed inside one process) and releases that
// rank's counter at system scope -- hand-over granularity is a column block (<= 62 KB), there is
// no kernel boundary, no staging copy and no NCCL call between steps.  The counters only ever
// grow (uses of a column block so far), so launches of different ranks need no alignment.
// ------------------------------------------------------------------------------------------
struct mfrec_ring {
    mfrec_ctx *ctx = nullptr;
    const mfrec_ratings *r = nullptr;
    mfrec_model *m = nullptr;
    int rank = 0, world = 1;
    // one cudaMalloc block (cudaIpcGetMemHandle exports whole allocations):
    //   [ Q  ni x kpad float | ib  ni float (padded) | ticks  G*B int32 | abort int32 ]
    char *block = nullptr;
    size_t off_ib = 0, off_ticks = 0, off_abort = 0, bytes = 0;
    char *peer = nullptr;        // the block of rank - 1 (the next user of every slab this rank finishes)
    bool peer_ipc = false;
    int64_t epochs_done = 0;
    double *se_part = nullptr;   // [epochs][B]
    size_t se_cap = 0;
    SgdRank *d_rank = nullptr;   // device copy of this rank's arguments
};

static float *ring_Q(char *b) { return reinterpret_cast<float *>(b); }

extern "C" void mfrec_ring_destroy(mfrec_ring *g)
{
    if (!g) return;
    cudaSetDevice(g->ctx->device);
    cudaStreamSynchronize(g->ctx->stream);
    if (g->peer && g->peer_ipc) cudaIpcCloseMemHandle(g->peer);
    if (g->block) cudaFree(g->block);
    if (g->se_part) cudaFree(g->se_part);
    if (g->d_rank) cudaFree(g->d_rank);
    mfrec_ctx_release(g->ctx);
    delete g;
}

extern "C" int mfrec_ring_create(mfrec_ctx *ctx, const mfrec_ratings *r, mfrec_model *m, int rank, int world,
                                 mfrec_ring **out)
{
    if (!ctx || !r || !m || !out) return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_ring_create: NULL argument");
    *out = nullptr;
    if (world < 1 || rank < 0 || rank >= world || r->G != world)
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_ring_create: rank %d of %d, layout has %d slabs (pack with n_slabs = world)",
                               rank, world, r->G);
    if (m->ni != r->ni || m->nu != r->nu || !m->user_perm || m->ni_rows != r->ni_v)
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_ring_create: model was not created with this layout");
    if (m->p_kind != MFREC_STORAGE_F32)
        return mfrec_set_error(ctx, MFREC_ERR_UNSUPPORTED, "mfrec_ring_create: the ring trains float32 user factors (opts.storage = 0)");
    MF_CUDA(ctx, cudaSetDevice(ctx->device));
    mfrec_ring *g = new (std::nothrow) mfrec_ring();
    if (!g) return mfrec_set_error(ctx, MFREC_ERR_OOM, "mfrec_ring_create: host OOM");
    g->ctx = ctx;
    mfrec_ctx_retain(ctx);
    g->r = r; g->m = m; g->rank = rank; g->world = world;
    const size_t qbytes = ((size_t)m->ni_rows * m->kpad + 64) * 4;
    g->off_ib = (qbytes + 255) & ~(size_t)255;
    g->off_ticks = (g->off_ib + ((size_t)m->ni_rows + 64) * 4 + 255) & ~(size_t)255;
    g->off_abort = g->off_ticks + (size_t)r->G * r->B * 4;
    g->bytes = g->off_abort + 256;
    struct Guard { mfrec_ring *g; ~Guard() { if (g) mfrec_ring_destroy(g); } } guard{g};
    MF_CUDA(ctx, cudaMalloc((void **)&g->block, g->bytes));
    MF_CUDA(ctx, cudaMalloc((void **)&g->d_rank, sizeof(SgdRank)));
    cudaStream_t st = ctx->stream;
    MF_CUDA(ctx, cudaMemsetAsync(g->block, 0, g->bytes, st));
    MF_CUDA(ctx, cudaMemcpyAsync(g->block, m->Q, (size_t)m->ni_rows * m->kpad * 4, cudaMemcpyDeviceToDevice, st));
    MF_CUDA(ctx, cudaMemcpyAsync(g->block + g->off_ib, m->ib, (size_t)m->ni_rows * 4, cudaMemcpyDeviceToDevice, st));
    MF_CUDA(ctx, cudaStreamSynchronize(st));
    guard.g = nullptr;
    *out = g;
    return MFREC_OK;
}

extern "C" int mfrec_ring_handle(mfrec_ring *g, void *handle64)
{
    if (!g || !handle64) return mfrec_set_error(g ? g->ctx : nullptr, MFREC_ERR_BAD_ARG, "mfrec_ring_handle: NULL argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size");
    MF_CUDA(g->ctx, cudaSetDevice(g->ctx->device));
    cudaIpcMemHandle_t h;
    MF_CUDA(g->ctx, cudaIpcGetMemHandle(&h, g->block));
    memcpy(handle64, &h, 64);
    return MFREC_OK;
}

extern "C" int mfrec_ring_connect(mfrec_ring *g, const void *handles)
{
    if (!g || (!handles && g->world > 1))
        return mfrec_set_error(g ? g->ctx : nullptr, MFREC_ERR_BAD_ARG, "mfrec_ring_connect: NULL argument");
    MF_CUDA(g->ctx, cudaSetDevice(g->ctx->device));
    if (g->world == 1) { g->peer = g->block; g->peer_ipc = false; return MFREC_OK; }
    const int dst = (g->rank + g->world - 1) % g->world;
    cudaIpcMemHandle_t h;
    memcpy(&h, static_cast<const char *>(handles) + (size_t)dst * 64, 64);
    void *p = nullptr;
    MF_CUDA(g->ctx, cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    g->peer = static_cast<char *>(p);
    g->peer_ipc = true;
    return MFREC_OK;
}

extern "C" int mfrec_ring_connect_local(mfrec_ring *g, mfrec_ring *next)
{
    if (!g || !next) return mfrec_set_error(g ? g->ctx : nullptr, MFREC_ERR_BAD_ARG, "mfrec_ring_connect_local: NULL argument");
    if (next->bytes != g->bytes || next->world != g->world || next->rank != (g->rank + g->world - 1) % g->world)
        return mfrec_set_error(g->ctx, MFREC_ERR_BAD_ARG, "mfrec_ring_connect_local: rank %d hands its slabs to rank %d, got rank %d",
                               g->rank, (g->rank + g->world - 1) % g->world, next->rank);
    MF_CUDA(g->ctx, cudaSetDevice(g->ctx->device));
    if (next->ctx->device != g->ctx->device) {
        int can = 0;
        MF_CUDA(g->ctx, cudaDeviceCanAccessPeer(&can, g->ctx->device, next->ctx->device));
        if (!can)
            return mfrec_set_error(g->ctx, MFREC_ERR_UNSUPPORTED, "device %d cannot address device %d", g->ctx->device, next->ctx->device);
        cudaError_t e = cudaDeviceEnablePeerAccess(next->ctx->device, 0);
        if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
        else MF_CUDA(g->ctx, e);
    }
    g->peer = next->block;
    g->peer_ipc = false;
    return MFREC_OK;
}

namespace {

void ring_rank_args(const mfrec_ring *g, SgdRank &a, double *se_part)
{
    a.packed = g->r->packed;
    a.bucket_off = g->r->bucket_off;
    a.col_start = g->r->col_start;
    a.Q = ring_Q(g->block);
    a.ib = reinterpret_cast<float *>(g->block + g->off_ib);
    a.P = g->m->P;
    a.ub = g->m->ub;
    a.se_part = se_part;
    a.ticks = reinterpret_cast<int32_t *>(g->block + g->off_ticks);
    a.peer_Q = ring_Q(g->peer);
    a.peer_ib = reinterpret_cast<float *>(g->peer + g->off_ib);
    a.peer_ticks = reinterpret_cast<int32_t *>(g->peer + g->off_ticks);
    a.abort = reinterpret_cast<int32_t *>(g->block + g->off_abort);
    a.rank = g->rank;
}

unsigned long long ring_wait_ns()
{
    const char *s = getenv("MFREC_RING_TIMEOUT_MS");
    return (unsigned long long)(s ? atoll(s) : 20000) * 1000000ull;
}

// out[e] = sum of the `n` partials of epoch e
__global__ void __launch_bounds__(256) se_reduce_epochs_kernel(const double *__restrict__ part, int n,
                                                               double *__restrict__ out)
{
    __shared__ double sh[256];
    const double *p = part + (size_t)blockIdx.x * n;
    double acc = 0.0;
    for (int i = threadIdx.x; i < n; i += 256) acc += p[i];
    sh[threadIdx.x] = acc;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) out[blockIdx.x] = sh[0];
}

// one launch over `n_ranks` rings that live on ONE device (n_ranks == 1: the normal case)
int ring_launch(mfrec_ring *const *rings, int n_ranks, int kernel, double learning_rate, double K_users,
                double K_items, double K_bias, int n_epochs, double *sq_err_out)
{
    mfrec_ring *g0 = rings[0];
    mfrec_ctx *ctx = g0->ctx;
    const mfrec_ratings *r = g0->r;
    if (n_epochs <= 0) return MFREC_OK;
    if (kernel != MFREC_KERNEL_LINEAR && kernel != MFREC_KERNEL_LOGISTIC)
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_ring_epochs: kernel=%d", kernel);
    for (int i = 0; i < n_ranks; ++i) {
        mfrec_ring *g = rings[i];
        if (!g->peer) return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_ring_epochs: rank %d is not connected", g->rank);
        if (g->ctx != ctx || g->r->B != r->B || g->r->W != r->W || g->r->G != r->G || g->m->kpad != g0->m->kpad ||
            g->r->max_cb_items != r->max_cb_items || g->epochs_done != g0->epochs_done)
            return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_ring_epochs: the rings of one launch must share context and layout shape");
    }
    MF_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t smem = mfrec_sgd_smem_bytes(r->max_cb_items, g0->m->kpad, r->W, 4);
    const int grid = n_ranks * r->B;
    if (smem > ctx->smem_optin || !ctx->coop_launch || !sgd_fits_one_wave(ctx, grid, r->W, smem))
        return mfrec_set_error(ctx, MFREC_ERR_UNSUPPORTED,
                               "mfrec_ring_epochs: %d CTAs x %zu B shared memory cannot be co-resident; pack with fewer row_blocks",
                               grid, smem);
    const size_t need = (size_t)n_epochs * grid;
    if (g0->se_cap < need) {
        if (g0->se_part) cudaFree(g0->se_part);
        g0->se_part = nullptr;
        g0->se_cap = 0;
        MF_CUDA(ctx, cudaMalloc((void **)&g0->se_part, need * 8));
        g0->se_cap = need;
    }
    bool hot = false;
    for (int i = 0; i < n_ranks; ++i) hot = hot || rings[i]->m->n_hot > 0;
    // layouts with hot-item copies merge them after every epoch: one launch per epoch (each rank's
    // merge waits for its neighbour's last pushes, so the next launch starts from merged rows)
    const int per_launch = hot ? 1 : n_epochs;
    const int64_t per_epoch = (int64_t)r->G * r->B;
    // Per-rank arguments: uploaded ONCE per call, before the first launch.  (A host -> device copy
    // between launches would be ordered behind the running kernel, and a process that drives several
    // devices would block in it before it has launched the neighbours that kernel is waiting for.)
    DevBuf<SgdRank> d_multi;
    SgdRank *d_args = g0->d_rank;
    {
        std::vector<SgdRank> args(n_ranks);
        for (int i = 0; i < n_ranks; ++i) ring_rank_args(rings[i], args[i], g0->se_part + (size_t)i * r->B);
        if (n_ranks > 1) {
            MF_CUDA(ctx, d_multi.alloc(n_ranks, ctx->stream));
            d_args = d_multi.p;
        }
        MF_CUDA(ctx, cudaMemcpyAsync(d_args, args.data(), sizeof(SgdRank) * n_ranks, cudaMemcpyHostToDevice, ctx->stream));
    }
    const int64_t e_first = g0->epochs_done;
    for (int e0 = 0; e0 < n_epochs; e0 += per_launch) {
        SgdParams prm;
        memset(&prm, 0, sizeof(prm));
        fill_hyper(prm, r, learning_rate, K_users, K_items, K_bias, 1, 1);
        prm.ranks = d_args;
        prm.B = r->B; prm.W = r->W; prm.G = r->G; prm.world = g0->world;
        prm.tile_rows = r->max_cb_items;
        prm.it_begin = g0->epochs_done * per_epoch;
        prm.it_end = (g0->epochs_done + per_launch) * per_epoch;
        prm.e_base = e_first;          // sums of epoch e go to se_part[(e - e_first) * grid ...]
        prm.se_stride = grid;
        prm.wait_ns = ring_wait_ns();
        MF_TRY(launch_sgd_kpad(ctx, g0->m->kpad, kernel, prm, smem, true, grid, true));
        for (int i = 0; i < n_ranks; ++i) rings[i]->epochs_done += per_launch;
        if (hot) {
            for (int i = 0; i < n_ranks; ++i) {
                mfrec_ring *g = rings[i];
                // after whole epochs rank i holds slab i: rows [a, b), column blocks [i * B, i * B + B)
                const int32_t a = g->r->h_col_start[(size_t)g->rank * r->B * r->W];
                const int32_t b = g->r->h_col_start[(size_t)(g->rank + 1) * r->B * r->W];
                const bool remote = g->world > 1 && n_ranks == 1;   // the pushes come from another device
                MF_TRY(mfrec_merge_copies(ctx, ring_Q(g->block), reinterpret_cast<float *>(g->block + g->off_ib), g->m->kpad,
                                          g->m->hot_off, g->m->hot_rows, g->m->n_hot, a, b,
                                          remote ? reinterpret_cast<const int32_t *>(g->block + g->off_ticks) : nullptr,
                                          g->rank * r->B, g->rank * r->B + r->B, (int32_t)(g->epochs_done * per_epoch),
                                          reinterpret_cast<int32_t *>(g->block + g->off_abort), ring_wait_ns()));
            }
        }
    }
    if (n_ranks > 1) MF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));   // d_multi is freed on return
    if (sq_err_out) {
        se_reduce_epochs_kernel<<<n_epochs, 256, 0, ctx->stream>>>(g0->se_part, grid, sq_err_out);
        MF_LAUNCH_CHECK(ctx);
    }
    return MFREC_OK;
}

}  // namespace

extern "C" int mfrec_ring_epochs(mfrec_ring *g, int kernel, double learning_rate, double K_users, double K_items,
                                 double K_bias, int n_epochs, double *sq_err_out)
{
    if (!g) return mfrec_set_error(nullptr, MFREC_ERR_BAD_ARG, "mfrec_ring_epochs: NULL ring");
    return ring_launch(&g, 1, kernel, learning_rate, K_users, K_items, K_bias, n_epochs, sq_err_out);
}

extern "C" int mfrec_ring_epochs_one_device(mfrec_ring *const *rings, int world, int kernel, double learning_rate,
                                            double K_users, double K_items, double K_bias, int n_epochs,
                                            double *sq_err_out)
{
    if (!rings || world < 1 || !rings[0])
        return mfrec_set_error(nullptr, MFREC_ERR_BAD_ARG, "mfrec_ring_epochs_one_device: NULL argument");
    for (int i = 0; i < world; ++i)
        if (!rings[i] || rings[i]->rank != i || rings[i]->world != world)
            return mfrec_set_error(rings[0]->ctx, MFREC_ERR_BAD_ARG, "mfrec_ring_epochs_one_device: rings[i] must be rank i of %d", world);
    return ring_launch(rings, world, kernel, learning_rate, K_users, K_items, K_bias, n_epochs, sq_err_out);
}

extern "C" int mfrec_ring_wait(mfrec_ring *g)
{
    if (!g) return mfrec_set_error(nullptr, MFREC_ERR_BAD_ARG, "mfrec_ring_wait: NULL ring");
    MF_CUDA(g->ctx, cudaSetDevice(g->ctx->device));
    int32_t ab = 0;
    MF_CUDA(g->ctx, cudaMemcpyAsync(&ab, g->block + g->off_abort, 4, cudaMemcpyDeviceToHost, g->ctx->stream));
    MF_CUDA(g->ctx, cudaStreamSynchronize(g->ctx->stream));
    if (ab)
        return mfrec_set_error(g->ctx, MFREC_ERR_CUDA,
                               "mfrec_ring_wait: rank %d gave up waiting for a column block from its neighbour (MFREC_RING_TIMEOUT_MS)",
                               g->rank);
    return MFREC_OK;
}

extern "C" int mfrec_ring_sync_model(mfrec_ring *g)
{
    if (!g) return mfrec_set_error(nullptr, MFREC_ERR_BAD_ARG, "mfrec_ring_sync_model: NULL ring");
    MF_TRY(mfrec_ring_wait(g));
    cudaStream_t st = g->ctx->stream;
    const mfrec_model *m = g->m;
    MF_CUDA(g->ctx, cudaMemcpyAsync(m->Q, g->block, (size_t)m->ni_rows * m->kpad * 4, cudaMemcpyDeviceToDevice, st));
    MF_CUDA(g->ctx, cudaMemcpyAsync(m->ib, g->block + g->off_ib, (size_t)m->ni_rows * 4, cudaMemcpyDeviceToDevice, st));
    MF_CUDA(g->ctx, cudaStreamSynchronize(st));
    return MFREC_OK;
}

static int train_kmf_sequential(mfrec_ctx *ctx, int kernel, int nbr_epochs, int k, double lr,
                                double K_users, double K_items, double K_bias, double *u, double *v,
                                const int32_t *idx, const double *ratings, int64_t nnz, int32_t ni,
                                int32_t nu, double *ib, double *ub, int update_users,
                                int update_items, double *rmse_per_epoch)
{
    cudaStream_t st = ctx->stream;
    DevBuf<double> du, dv, dr, dib, dub, drm;
    DevBuf<int32_t> didx;
    MF_CUDA(ctx, du.alloc((size_t)k * ni, ctx->stream));
    MF_CUDA(ctx, dv.alloc((size_t)k * nu, ctx->stream));
    MF_CUDA(ctx, dr.alloc((size_t)nnz, ctx->stream));
    MF_CUDA(ctx, didx.alloc((size_t)nnz * 2, ctx->stream));
    MF_CUDA(ctx, dib.alloc(ni, ctx->stream));
    MF_CUDA(ctx, dub.alloc(nu, ctx->stream));
    MF_CUDA(ctx, drm.alloc(nbr_epochs > 0 ? nbr_epochs : 1, ctx->stream));
    MF_CUDA(ctx, cudaMemcpyAsync(du.p, u, (size_t)k * ni * 8, cudaMemcpyHostToDevice, st));
    MF_CUDA(ctx, cudaMemcpyAsync(dv.p, v, (size_t)k * nu * 8, cudaMemcpyHostToDevice, st));
    MF_CUDA(ctx, cudaMemcpyAsync(dr.p, ratings, (size_t)nnz * 8, cudaMemcpyHostToDevice, st));
    MF_CUDA(ctx, cudaMemcpyAsync(didx.p, idx, (size_t)nnz * 8, cudaMemcpyHostToDevice, st));
    MF_CUDA(ctx, cudaMemcpyAsync(dib.p, ib, (size_t)ni * 8, cudaMemcpyHostToDevice, st));
    MF_CUDA(ctx, cudaMemcpyAsync(dub.p, ub, (size_t)nu * 8, cudaMemcpyHostToDevice, st));
    kmf_sequential_kernel<<<1, 32, 0, st>>>(kernel, nbr_epochs, k, lr, K_users, K_items, K_bias, du.p,
                                           dv.p, didx.p, dr.p, nnz, ni, nu, dib.p, dub.p,
                                           update_users, update_items, drm.p);
    MF_LAUNCH_CHECK(ctx);
    MF_CUDA(ctx, cudaMemcpyAsync(u, du.p, (size_t)k * ni * 8, cudaMemcpyDeviceToHost, st));
    MF_CUDA(ctx, cudaMemcpyAsync(v, dv.p, (size_t)k * nu * 8, cudaMemcpyDeviceToHost, st));
    MF_CUDA(ctx, cudaMemcpyAsync(ib, dib.p, (size_t)ni * 8, cudaMemcpyDeviceToHost, st));
    MF_CUDA(ctx, cudaMemcpyAsync(ub, dub.p, (size_t)nu * 8, cudaMemcpyDeviceToHost, st));
    if (rmse_per_epoch && nbr_epochs > 0)
        MF_CUDA(ctx, cudaMemcpyAsync(rmse_per_epoch, drm.p, (size_t)nbr_epochs * 8, cudaMemcpyDeviceToHost, st));
    MF_CUDA(ctx, cudaStreamSynchronize(st));
    return MFREC_OK;
}

extern "C" int mfrec_train_kmf(mfrec_ctx *ctx, int kernel, int nbr_epochs, int k, double learning_rate,
                               double K_users, double K_items, double K_bias, double *u, double *v,
                               const int32_t *ratings_index, const double *ratings, int64_t nnz,
                               int32_t ni, int32_t nu, double *items_bias, double *users_bias,
                               int update_users, int update_items, const mfrec_opts *opts,
                               double *rmse_per_epoch)
{
    if (!ctx) return mfrec_set_error(nullptr, MFREC_ERR_BAD_ARG, "mfrec_train_kmf: NULL ctx");
    if (!u || !v || !items_bias || !users_bias || (nnz > 0 && (!ratings_index || !ratings)))
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_train_kmf: NULL array");
    if (kernel != MFREC_KERNEL_LINEAR && kernel != MFREC_KERNEL_LOGISTIC)
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_train_kmf: kernel=%d", kernel);
    if (k <= 0 || ni <= 0 || nu <= 0 || nnz < 0 || nbr_epochs < 0)
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_train_kmf: k=%d ni=%d nu=%d nnz=%lld epochs=%d",
                               k, ni, nu, (long long)nnz, nbr_epochs);
    MF_CUDA(ctx, cudaSetDevice(ctx->device));
    if (nbr_epochs == 0) return MFREC_OK;
    if (nnz == 0) {
        // the reference divides 0/0 -> rmse = NaN and leaves the model untouched
        if (rmse_per_epoch)
            for (int e = 0; e < nbr_epochs; ++e) rmse_per_epoch[e] = NAN;
        return MFREC_OK;
    }
    if (opts && opts->schedule == MFREC_SCHED_SEQUENTIAL) {
        for (int64_t n = 0; n < nnz; ++n) {
            const int32_t a = ratings_index[2 * n], b = ratings_index[2 * n + 1];
            if (a < 0 || a >= nu || b < 0 || b >= ni)
                return mfrec_set_error(ctx, MFREC_ERR_INDEX, "mfrec_train_kmf: rating %lld has (user,item)=(%d,%d)",
                                       (long long)n, a, b);
        }
        // A fold-in (KMFRecommender.retrain_user / retrain_item / add_user, kmf.py:120-172) names a
        // handful of rows: move only those (FoldRows).
        if (nnz <= 65536 && (int64_t)ni + nu > 4 * nnz) {
            FoldRows g;
            g.gather(k, false, u, v, items_bias, users_bias, ni, nu, ratings_index, nnz);
            MF_TRY(train_kmf_sequential(ctx, kernel, nbr_epochs, k, learning_rate, K_users, K_items, K_bias,
                                        g.u.data(), g.v.data(), g.idx.data(), ratings, nnz, (int32_t)g.items.size(),
                                        (int32_t)g.users.size(), g.ib.data(), g.ub.data(), update_users,
                                        update_items, rmse_per_epoch));
            g.scatter(u, v, items_bias, users_bias, ni, nu);
            return MFREC_OK;
        }
        return train_kmf_sequential(ctx, kernel, nbr_epochs, k, learning_rate, K_users, K_items, K_bias,
                                    u, v, ratings_index, ratings, nnz, ni, nu, items_bias, users_bias,
                                    update_users, update_items, rmse_per_epoch);
    }
    if (mfrec_kpad(k) < 0)
        return mfrec_set_error(ctx, MFREC_ERR_UNSUPPORTED, "mfrec_train_kmf: k=%d > 256 is not instantiated", k);
    mfrec_opts o;
    if (opts) o = *opts; else memset(&o, 0, sizeof(o));
    o.n_slabs = 1;
    if (o.k_hint == 0) o.k_hint = k;
    mfrec_ratings *R = nullptr;
    mfrec_model *M = nullptr;
    Tracer tr("train_kmf", ctx->stream);
    // Host -> device: the index array goes first on the context stream, so the packer can start
    // (degrees, partition, sort) while the rating values and the float64 factor arrays are still
    // crossing PCIe on the copy stream; the packer's gather and the layout conversion wait for
    // their events.
    cudaStream_t sa = ctx->stream, sb = ctx->copy_stream;
    DevBuf<int32_t> d_idx;
    DevBuf<double> d_r, d_u, d_v, d_ib, d_ub;
    cudaEvent_t ev_idx = nullptr, ev_val = nullptr, ev_fac = nullptr;
    struct EvGuard {
        cudaEvent_t *e[3];
        mfrec_ctx *c;
        ~EvGuard()
        {
            c->values_ready = nullptr;
            c->staged = {};
            cudaStreamSynchronize(c->copy_stream);   // nothing may still write the staging buffers
            for (auto p : e) if (*p) cudaEventDestroy(*p);
        }
    } evg{{&ev_idx, &ev_val, &ev_fac}, ctx};
    MF_CUDA(ctx, cudaEventCreateWithFlags(&ev_idx, cudaEventDisableTiming));
    MF_CUDA(ctx, cudaEventCreateWithFlags(&ev_val, cudaEventDisableTiming));
    MF_CUDA(ctx, cudaEventCreateWithFlags(&ev_fac, cudaEventDisableTiming));
    MF_CUDA(ctx, d_idx.alloc((size_t)nnz * 2, sa));
    MF_CUDA(ctx, d_r.alloc((size_t)nnz, sa));
    MF_CUDA(ctx, d_u.alloc((size_t)k * ni, sa));
    MF_CUDA(ctx, d_v.alloc((size_t)k * nu, sa));
    MF_CUDA(ctx, d_ib.alloc(ni, sa));
    MF_CUDA(ctx, d_ub.alloc(nu, sa));
    // the two small bias arrays first: callers often keep them in pageable memory, and a pageable
    // copy blocks the host until everything queued before it on its stream has drained
    MF_CUDA(ctx, cudaMemcpyAsync(d_ib.p, items_bias, (size_t)ni * 8, cudaMemcpyHostToDevice, sa));
    MF_CUDA(ctx, cudaMemcpyAsync(d_ub.p, users_bias, (size_t)nu * 8, cudaMemcpyHostToDevice, sa));
    // (mfrec_copy_h2d: page-locked arrays go straight to cudaMemcpyAsync and everything below
    // overlaps with the packer; large pageable arrays are staged by four host threads first)
    MF_TRY(mfrec_copy_h2d(ctx, d_idx.p, ratings_index, (size_t)nnz * 8, sa));
    MF_CUDA(ctx, cudaEventRecord(ev_idx, sa));
    MF_CUDA(ctx, cudaStreamWaitEvent(sb, ev_idx, 0));   // (also orders the pool allocations before sb's use)
    // The remaining uploads on the copy stream.  Page-locked arrays: four asynchronous copies, this
    // thread goes straight on to the packer.  Pageable arrays are staged through bounce buffers by
    // host threads, which blocks the caller: a background thread does it, so the packer (which needs
    // the values only for its last step, and the factors not at all) still overlaps with the upload.
    auto upload_rest = [&](std::promise<int> *p_val, std::promise<int> *p_fac) -> int {
        int urc = mfrec_copy_h2d(ctx, d_r.p, ratings, (size_t)nnz * 8, sb);
        if (urc == MFREC_OK && cudaEventRecord(ev_val, sb) != cudaSuccess)
            urc = mfrec_set_error(ctx, MFREC_ERR_CUDA, "mfrec_train_kmf: cudaEventRecord failed");
        if (p_val) p_val->set_value(urc);
        if (urc == MFREC_OK) urc = mfrec_copy_h2d(ctx, d_v.p, v, (size_t)k * nu * 8, sb);
        if (urc == MFREC_OK) urc = mfrec_copy_h2d(ctx, d_u.p, u, (size_t)k * ni * 8, sb);
        if (urc == MFREC_OK && cudaEventRecord(ev_fac, sb) != cudaSuccess)
            urc = mfrec_set_error(ctx, MFREC_ERR_CUDA, "mfrec_train_kmf: cudaEventRecord failed");
        if (p_fac) p_fac->set_value(urc);
        return urc;
    };
    std::promise<int> p_val, p_fac;
    struct UploadThread {
        std::thread t;
        mfrec_ctx *c;
        ~UploadThread()
        {
            if (t.joinable()) t.join();
            c->values_enqueued = {};
            c->factors_enqueued = {};
        }
    } up{{}, ctx};
    if (mfrec_host_needs_staging(ratings, (size_t)nnz * 8) || mfrec_host_needs_staging(v, (size_t)k * nu * 8) ||
        mfrec_host_needs_staging(u, (size_t)k * ni * 8)) {
        ctx->values_enqueued = p_val.get_future().share();
        ctx->factors_enqueued = p_fac.get_future().share();
        const int device = ctx->device;
        up.t = std::thread([&upload_rest, &p_val, &p_fac, device]() {
            cudaSetDevice(device);
            upload_rest(&p_val, &p_fac);
        });
    } else {
        MF_TRY(upload_rest(nullptr, nullptr));
    }
    ctx->values_ready = ev_val;
    MF_TRY(mfrec_ratings_pack(ctx, d_idx.p, d_r.p, 0, 1, nnz, ni, nu, nullptr, &o, &R));
    tr.lap("pack");
    ctx->staged.u = d_u.p; ctx->staged.v = d_v.p; ctx->staged.ib = d_ib.p; ctx->staged.ub = d_ub.p;
    ctx->staged.ready = ev_fac;
    int rc = mfrec_model_create(ctx, R, k, ni, nu, u, v, items_bias, users_bias, &M);
    if (rc == MFREC_OK) {   // the staging buffers go back to the pool on sa: sb must be done with them
        cudaError_t we = cudaStreamWaitEvent(sa, ev_fac, 0);
        if (we != cudaSuccess) rc = mfrec_set_error(ctx, MFREC_ERR_CUDA, "cudaStreamWaitEvent: %s", cudaGetErrorString(we));
    } else {
        cudaStreamSynchronize(sb);
    }
    tr.lap("model upload");
    DevBuf<double> d_se;
    if (rc == MFREC_OK && d_se.alloc(nbr_epochs, ctx->stream) != cudaSuccess)
        rc = mfrec_set_error(ctx, MFREC_ERR_OOM, "mfrec_train_kmf: device OOM");
    for (int e = 0; rc == MFREC_OK && e < nbr_epochs; ++e)
        rc = mfrec_sgd_epoch(ctx, R, M, kernel, learning_rate, K_users, K_items, K_bias, update_users,
                             update_items, -1, d_se.p + e);
    if (rc == MFREC_OK) {
        std::vector<double> h_se(nbr_epochs);
        cudaError_t ce = cudaMemcpyAsync(h_se.data(), d_se.p, (size_t)nbr_epochs * 8, cudaMemcpyDeviceToHost, ctx->stream);
        if (ce == cudaSuccess) ce = cudaStreamSynchronize(ctx->stream);
        if (ce != cudaSuccess) rc = mfrec_set_error(ctx, MFREC_ERR_CUDA, "mfrec_train_kmf: %s", cudaGetErrorString(ce));
        else if (rmse_per_epoch)
            for (int e = 0; e < nbr_epochs; ++e) rmse_per_epoch[e] = sqrt(h_se[e] / (double)nnz);
    }
    tr.lap("epochs");
    if (rc == MFREC_OK) rc = mfrec_model_read(ctx, M, u, v, items_bias, users_bias);
    tr.lap("model download");
    mfrec_model_destroy(M);
    mfrec_ratings_destroy(R);
    tr.lap("free");
    return rc;
}

extern "C" int mfrec_fold_in_kmf(mfrec_ctx *ctx, int kernel, int side, int nbr_epochs, int k, double learning_rate,
                                 double K_users, double K_items, double K_bias, double *u, double *v,
                                 const int32_t *ratings_index, const double *ratings, int64_t nnz,
                                 int32_t ni, int32_t nu, double *items_bias, double *users_bias,
                                 const int32_t *rows, int32_t n_rows, double *rmse)
{
    if (!ctx) return mfrec_set_error(nullptr, MFREC_ERR_BAD_ARG, "mfrec_fold_in_kmf: NULL ctx");
    if (!u || !v || !items_bias || !users_bias || (nnz > 0 && (!ratings_index || !ratings)) || (n_rows > 0 && !rows))
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_fold_in_kmf: NULL array");
    if (kernel != MFREC_KERNEL_LINEAR && kernel != MFREC_KERNEL_LOGISTIC)
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_fold_in_kmf: kernel=%d", kernel);
    if (side != MFREC_FOLD_USERS && side != MFREC_FOLD_ITEMS)
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_fold_in_kmf: side=%d", side);
    if (k <= 0 || ni <= 0 || nu <= 0 || nnz < 0 || nbr_epochs < 0 || n_rows < 0)
        return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "mfrec_fold_in_kmf: k=%d ni=%d nu=%d nnz=%lld epochs=%d rows=%d",
                               k, ni, nu, (long long)nnz, nbr_epochs, n_rows);
    const bool by_user = side == MFREC_FOLD_USERS, linear = kernel == MFREC_KERNEL_LINEAR;
    const int tc = by_user ? 0 : 1;   // column of ratings_index naming the trained row; 1 - tc the frozen one
    FoldSelection sel;
    MF_TRY(sel.count(ctx, "mfrec_fold_in_kmf", side, ratings_index, nnz, ni, nu, rows, n_rows));
    const std::vector<int64_t> &rptr = sel.rptr;
    const int64_t nsel = sel.nsel();
    MF_CUDA(ctx, cudaSetDevice(ctx->device));
    if (nbr_epochs == 0) return MFREC_OK;
    if (rmse)   // a row without ratings: the reference divides 0/0 and leaves the model untouched
        for (int32_t p = 0; p < n_rows; ++p)
            if (rptr[p + 1] == rptr[p])
                for (int e = 0; e < nbr_epochs; ++e) rmse[(size_t)p * nbr_epochs + e] = NAN;
    if (nsel == 0) return MFREC_OK;
    sel.gather(ratings_index, ratings, nnz);
    const std::vector<double> &sr = sel.r;
    // the listed rows and the frozen rows their ratings name, row-major (a lane reads whole rows)
    FoldRows g;
    g.gather(k, true, u, v, items_bias, users_bias, ni, nu, sel.idx.data(), nsel);
    std::vector<double> &tf = by_user ? g.v : g.u, &tb = by_user ? g.ub : g.ib, &fbv = by_user ? g.ib : g.ub;
    const std::vector<double> &ff = by_user ? g.u : g.v;
    const size_t n_frozen = by_user ? g.items.size() : g.users.size();

    // Levels.  Logistic: rows share no written state, one level.  Linear: a row's ratings write the
    // biases of its frozen rows, so a row runs after every earlier listed row that shares a frozen
    // row with it: level = 1 + the highest level of such a row (one "last level" per frozen row).
    struct Job { int32_t level, p; int64_t cnt; };
    std::vector<Job> jobs;
    jobs.reserve(n_rows);
    std::vector<int32_t> last(linear ? n_frozen : 0, 0);
    for (int32_t p = 0; p < n_rows; ++p) {
        const int64_t a = rptr[p], b = rptr[p + 1];
        if (a == b) continue;
        int32_t level = 1;
        if (linear) {
            for (int64_t n = a; n < b; ++n) level = std::max(level, last[g.idx[2 * n + 1 - tc]] + 1);
            for (int64_t n = a; n < b; ++n) last[g.idx[2 * n + 1 - tc]] = level;
        }
        jobs.push_back({level, p, b - a});
    }
    // levels in order; inside a level the longest rows first, so the lanes of a warp have similar trip counts
    std::stable_sort(jobs.begin(), jobs.end(), [](const Job &x, const Job &y) {
        return x.level != y.level ? x.level < y.level : x.cnt > y.cnt;
    });
    const int32_t n_jobs = (int32_t)jobs.size();
    std::vector<int32_t> job_row(n_jobs), fidx(nsel), level_start;
    std::vector<int64_t> job_ptr((size_t)n_jobs + 1, 0);
    std::vector<double> rv(nsel);
    for (int32_t j = 0; j < n_jobs; ++j) {
        const Job &J = jobs[j];
        if (j == 0 || J.level != jobs[j - 1].level) level_start.push_back(j);
        const int64_t a = rptr[J.p];
        job_row[j] = g.idx[2 * a + tc];
        for (int64_t n = 0; n < J.cnt; ++n) {
            fidx[job_ptr[j] + n] = g.idx[2 * (a + n) + 1 - tc];
            rv[job_ptr[j] + n] = sr[a + n];
        }
        job_ptr[j + 1] = job_ptr[j] + J.cnt;
    }
    level_start.push_back(n_jobs);

    // lanes per block: as many per-lane shared-memory rows as fit (up to a warp)
    const size_t row_bytes = (size_t)k * 8;
    const int lanes = (int)std::min<size_t>(32, ctx->smem_optin / row_bytes);
    const bool smem = lanes > 0;
    const int block = smem ? lanes : 32;
    const size_t smem_bytes = smem ? (size_t)lanes * row_bytes : 0;
    auto launch = by_user ? (smem ? kmf_fold_in_kernel<true, MFREC_FOLD_USERS> : kmf_fold_in_kernel<false, MFREC_FOLD_USERS>)
                          : (smem ? kmf_fold_in_kernel<true, MFREC_FOLD_ITEMS> : kmf_fold_in_kernel<false, MFREC_FOLD_ITEMS>);
    if (smem_bytes > 48 * 1024)
        MF_CUDA(ctx, cudaFuncSetAttribute(launch, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));

    cudaStream_t st = ctx->stream;
    DevBuf<double> d_tf, d_tb, d_ff, d_fb, d_rv, d_rm;
    DevBuf<int32_t> d_row, d_fidx;
    DevBuf<int64_t> d_ptr;
    MF_CUDA(ctx, d_tf.alloc(tf.size(), st));
    MF_CUDA(ctx, d_tb.alloc(tb.size(), st));
    MF_CUDA(ctx, d_ff.alloc(ff.size(), st));
    MF_CUDA(ctx, d_fb.alloc(fbv.size(), st));
    MF_CUDA(ctx, d_rv.alloc(nsel, st));
    MF_CUDA(ctx, d_fidx.alloc(nsel, st));
    MF_CUDA(ctx, d_row.alloc(n_jobs, st));
    MF_CUDA(ctx, d_ptr.alloc((size_t)n_jobs + 1, st));
    MF_CUDA(ctx, d_rm.alloc((size_t)n_jobs * nbr_epochs, st));
    MF_CUDA(ctx, cudaMemcpyAsync(d_tf.p, tf.data(), tf.size() * 8, cudaMemcpyHostToDevice, st));
    MF_CUDA(ctx, cudaMemcpyAsync(d_tb.p, tb.data(), tb.size() * 8, cudaMemcpyHostToDevice, st));
    MF_CUDA(ctx, cudaMemcpyAsync(d_ff.p, ff.data(), ff.size() * 8, cudaMemcpyHostToDevice, st));
    MF_CUDA(ctx, cudaMemcpyAsync(d_fb.p, fbv.data(), fbv.size() * 8, cudaMemcpyHostToDevice, st));
    MF_CUDA(ctx, cudaMemcpyAsync(d_rv.p, rv.data(), (size_t)nsel * 8, cudaMemcpyHostToDevice, st));
    MF_CUDA(ctx, cudaMemcpyAsync(d_fidx.p, fidx.data(), (size_t)nsel * 4, cudaMemcpyHostToDevice, st));
    MF_CUDA(ctx, cudaMemcpyAsync(d_row.p, job_row.data(), (size_t)n_jobs * 4, cudaMemcpyHostToDevice, st));
    MF_CUDA(ctx, cudaMemcpyAsync(d_ptr.p, job_ptr.data(), ((size_t)n_jobs + 1) * 8, cudaMemcpyHostToDevice, st));
    for (size_t L = 0; L + 1 < level_start.size(); ++L) {
        const int32_t j0 = level_start[L], n = level_start[L + 1] - j0;
        const int grid = (n + block - 1) / block;
        launch<<<grid, block, smem_bytes, st>>>(kernel, nbr_epochs, k, learning_rate, K_users, K_items, K_bias,
                                                d_tf.p, d_tb.p, d_ff.p, d_fb.p, d_row.p + j0, d_ptr.p + j0, d_fidx.p,
                                                d_rv.p, n, d_rm.p + (size_t)j0 * nbr_epochs);
        MF_LAUNCH_CHECK(ctx);
    }
    std::vector<double> h_rm((size_t)n_jobs * nbr_epochs);
    MF_CUDA(ctx, cudaMemcpyAsync(tf.data(), d_tf.p, tf.size() * 8, cudaMemcpyDeviceToHost, st));
    MF_CUDA(ctx, cudaMemcpyAsync(tb.data(), d_tb.p, tb.size() * 8, cudaMemcpyDeviceToHost, st));
    if (linear) MF_CUDA(ctx, cudaMemcpyAsync(fbv.data(), d_fb.p, fbv.size() * 8, cudaMemcpyDeviceToHost, st));
    MF_CUDA(ctx, cudaMemcpyAsync(h_rm.data(), d_rm.p, h_rm.size() * 8, cudaMemcpyDeviceToHost, st));
    MF_CUDA(ctx, cudaStreamSynchronize(st));
    // only the trained side (and, linear, the frozen biases) goes back: the frozen rows and every
    // unlisted row are never written
    if (by_user) g.scatter(nullptr, v, linear ? items_bias : nullptr, users_bias, ni, nu);
    else g.scatter(u, nullptr, items_bias, linear ? users_bias : nullptr, ni, nu);
    if (rmse)
        for (int32_t j = 0; j < n_jobs; ++j)
            std::copy(h_rm.begin() + (size_t)j * nbr_epochs, h_rm.begin() + (size_t)(j + 1) * nbr_epochs,
                      rmse + (size_t)jobs[j].p * nbr_epochs);
    return MFREC_OK;
}
