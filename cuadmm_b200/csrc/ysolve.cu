// ysolve.cu — y = (A A^T + eps I)^-1 rhs on the device.
//
// Replaces the reference's per-iteration host path (src/solver.cu:487-500, 704-717):
//   perform_permutation -> cudaDeviceSynchronize -> D2H -> cholmod_solve2 (host, simplicial LDL^T)
//   -> H2D -> perform_permutation
// with: gather-permute fused into a level-scheduled sparse forward sweep, a dense GEMV pair on the
// explicitly inverted trailing block of the factor (where the elimination DAG degenerates into a
// chain), a sparse backward sweep with the scatter-permute fused in.  Nothing leaves the GPU and
// there is no host synchronisation.
#include "ysolve.h"
#include <chrono>
#include <thread>
#include <atomic>
#include "dense.h"
#include <algorithm>
#include <numeric>
#include <stdio.h>
#include <stdlib.h>

namespace cuadmm {

static constexpr int kTriThreads = 256;
static constexpr int kLongRowNnz = 24;     // rows with more dependencies get a whole warp
static constexpr int kNarrowSlots = 160;   // levels with at most this many warp-slots run inside one CTA
static constexpr int kNarrowThreads = 1024;

// Work of a triangular sweep is cut into warp-slots: a slot is either 8 short rows (4 lanes each) or
// 1 long row (32 lanes), all of one dependency level.  The levels are grouped into phases:
//   wide level   -> one launch of tri_wide_kernel, one warp per slot, the stream order is the barrier;
//   narrow run   -> consecutive narrow levels in ONE CTA (tri_narrow_kernel), __syncthreads between
//                   levels (~0.1 us instead of a ~2.5 us kernel boundary or a multi-us global counter
//                   handshake; the deep end of the elimination DAG is hundreds of levels a few rows wide).
// No spin-waiting anywhere, so no co-residency requirement and nothing to deadlock.
// Unknown u:  x[u] = (rhs[u] - sum_p val[p] * x[dep[p]]) * inv_diag[u].
// Everything of a slot that does not depend on x (structure, values, right-hand side) is loaded by
// SlotWork::load and can therefore be issued one level AHEAD of the level barrier; finish() then
// only has the x loads on its critical path.  The deep end of the elimination DAG is latency-bound:
// this turns a chain of five dependent global loads per level into one.
struct SlotWork {
    static constexpr int K = 4;        // entries per lane kept in registers
    int32_t u; int is_long;
    double rv, invd;
    int64_t p, p1; int step;
    int32_t d[K]; double v[K];

    __device__ __forceinline__ void load(int64_t s, int lane, const int32_t* __restrict__ slot_rows,
            const int32_t* __restrict__ slot_info, const int64_t* __restrict__ ptr, const int32_t* __restrict__ dep,
            const double* __restrict__ val, const double* __restrict__ inv_diag, const double* __restrict__ rhs,
            const int32_t* __restrict__ rhs_gather) {
        is_long = slot_info[s] >> 30;
        u = slot_rows[8 * s + (is_long ? 0 : (lane >> 2))];
        step = is_long ? 32 : 4;
        p = 0; p1 = 0; rv = 0.0; invd = 0.0;
        if (u >= 0) {
            p = ptr[u] + (is_long ? lane : (lane & 3));
            p1 = ptr[u + 1];
            invd = inv_diag[u];
            rv = rhs_gather ? rhs[rhs_gather[u]] : rhs[u];
        }
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const int64_t q = p + (int64_t)k * step;
            if (q < p1) { d[k] = dep[q]; v[k] = val[q]; } else { d[k] = -1; v[k] = 0.0; }
        }
    }
    __device__ __forceinline__ void finish(int lane, const int32_t* __restrict__ dep, const double* __restrict__ val,
                                           double* x, double* out_scatter, const int32_t* __restrict__ out_perm) {
        double acc = 0.0;
#pragma unroll
        for (int k = 0; k < K; ++k) if (d[k] >= 0) acc = fma(v[k], x[d[k]], acc);
        for (int64_t q = p + (int64_t)K * step; q < p1; q += step) acc = fma(val[q], x[dep[q]], acc);
        acc += __shfl_xor_sync(0xffffffffu, acc, 1);
        acc += __shfl_xor_sync(0xffffffffu, acc, 2);
        if (is_long) {
            acc += __shfl_xor_sync(0xffffffffu, acc, 4);
            acc += __shfl_xor_sync(0xffffffffu, acc, 8);
            acc += __shfl_xor_sync(0xffffffffu, acc, 16);
        }
        const bool writer = (u >= 0) && (is_long ? (lane == 0) : ((lane & 3) == 0));
        if (writer) {
            const double r = (rv - acc) * invd;
            x[u] = r;
            if (out_scatter) out_scatter[out_perm[u]] = r;
        }
    }
};

#define CUADMM_TRI_PARAMS                                                                                   \
    const int32_t* __restrict__ slot_rows, const int32_t* __restrict__ slot_info, const int64_t* __restrict__ ptr, \
    const int32_t* __restrict__ dep, const double* __restrict__ val, const double* __restrict__ inv_diag,   \
    const double* __restrict__ rhs, const int32_t* __restrict__ rhs_gather, double* x, double* out_scatter, \
    const int32_t* __restrict__ out_perm, const int* __restrict__ done_flag
#define CUADMM_TRI_LOAD(W, S) (W).load((S), lane, slot_rows, slot_info, ptr, dep, val, inv_diag, rhs, rhs_gather)
#define CUADMM_TRI_FINISH(W) (W).finish(lane, dep, val, x, out_scatter, out_perm)

__global__ void __launch_bounds__(kTriThreads) tri_wide_kernel(int64_t slot0, int64_t slot1, CUADMM_TRI_PARAMS) {
    if (done_flag && *done_flag) return;
    const int lane = threadIdx.x & 31;
    const int64_t s = slot0 + (((int64_t)blockIdx.x * kTriThreads + threadIdx.x) >> 5);
    if (s >= slot1) return;
    SlotWork w;
    CUADMM_TRI_LOAD(w, s);
    CUADMM_TRI_FINISH(w);
}

// levels [level0, level1) of lvl_ptr inside one CTA of NW warps; the first slot of the next level is
// prefetched (static part) before the barrier of the current one
template <int NW>
__device__ __forceinline__ void tri_level_loop(const int64_t* __restrict__ lvl_ptr, int level0, int level1, int lane, int warp,
        CUADMM_TRI_PARAMS) {
    (void)done_flag;
    if (level0 >= level1) return;
    SlotWork w;
    int64_t s0 = lvl_ptr[level0];
    int64_t s1 = lvl_ptr[level0 + 1];
    bool have = (s0 + warp) < s1;
    if (have) CUADMM_TRI_LOAD(w, s0 + warp);
    for (int l = level0; l < level1; ++l) {
        if (have) {
            CUADMM_TRI_FINISH(w);
            for (int64_t s = s0 + warp + NW; s < s1; s += NW) { SlotWork t; CUADMM_TRI_LOAD(t, s); CUADMM_TRI_FINISH(t); }
        }
        s0 = s1;
        have = false;
        if (l + 1 < level1) {
            s1 = lvl_ptr[l + 2];
            have = (s0 + warp) < s1;
            if (have) CUADMM_TRI_LOAD(w, s0 + warp);
        }
        __syncthreads();   // also makes this CTA's global writes visible to its own later loads
    }
}

__global__ void __launch_bounds__(kNarrowThreads) tri_narrow_kernel(int level0, int level1, const int64_t* __restrict__ level_ptr,
                                                                    CUADMM_TRI_PARAMS) {
    if (done_flag && *done_flag) return;
    tri_level_loop<kNarrowThreads / 32>(level_ptr, level0, level1, threadIdx.x & 31, threadIdx.x >> 5,
        slot_rows, slot_info, ptr, dep, val, inv_diag, rhs, rhs_gather, x, out_scatter, out_perm, done_flag);
}

// Subtree parallelism: every CTA owns one subtree of the elimination tree (all of whose dependencies
// are inside the subtree, or already final), and walks the subtree's own levels with __syncthreads.
// Thousands of independent deep chains (one per block neighbourhood of a moment relaxation) thus cost
// ONE launch and depth x (one x-load latency) instead of depth x (kernel boundary).
__global__ void __launch_bounds__(kTriThreads) tri_subtree_kernel(const int64_t* __restrict__ sub_off,
        const int64_t* __restrict__ sub_lvl_ptr, CUADMM_TRI_PARAMS) {
    if (done_flag && *done_flag) return;
    const int64_t base = sub_off[blockIdx.x];
    const int nl = (int)(sub_off[blockIdx.x + 1] - base) - 1;
    tri_level_loop<kTriThreads / 32>(sub_lvl_ptr + base, 0, nl, threadIdx.x & 31, threadIdx.x >> 5,
        slot_rows, slot_info, ptr, dep, val, inv_diag, rhs, rhs_gather, x, out_scatter, out_perm, done_flag);
}

// ---------------------------------------------------------------------------------------------
// Packed subtrees.  The x-independent data of a subtree (structure + values of its rows, already in
// level order) is laid out on the host as a stream of fixed-size CHUNKS, which one thread moves
// global -> shared with 1-D TMA bulk copies (cp.async.bulk + mbarrier) kPkRing chunks ahead of the
// warps that consume them.  Chunk size (measured on the bench problem, ms per solve): 8 KB x 6: 0.378, 16 KB x 4:
// 0.331, 32 KB x 3: 0.310, 48 KB x 3: 0.301, 64 KB x 2: 0.295 — every chunk boundary is a barrier on top of the
// level barriers, so the largest chunk that leaves room for the unknowns wins.  The unknowns live in shared memory for the whole kernel, so a level
// costs one __syncthreads plus shared-memory traffic: no global load sits on the critical path.
//
// chunk:  u16 nseg, u16 nslots, u16 seg_end[nseg], u16 rec_off[nslots] (8-byte units), records...
//         a segment = consecutive slots of one level; every segment ends with a barrier.
// record: i32 is_long, i32 ne, i32 slot[8], u16 voff[8] (8-byte units), u16 ioff[8] (2-byte units), u16 len[8],
//         f64 inv_diag[8], f64 val[ne], u16 idx[ne]
//         (8 short rows x 4 lanes, or one long row x 32 lanes; idx = shared-memory index of the dependency)
// Dependencies OUTSIDE the subtree are final when the kernel starts; the prologue folds them into
// the right-hand side:  xs[loc] = rhs[u] - sum_ext val * x[dep].
#ifndef CUADMM_PK_CHUNK
#define CUADMM_PK_CHUNK 65536
#endif
#ifndef CUADMM_PK_RING
#define CUADMM_PK_RING 2
#endif
static constexpr int kPkChunk = CUADMM_PK_CHUNK;
static constexpr int kPkRing = CUADMM_PK_RING;
#ifndef CUADMM_PK_THREADS
#define CUADMM_PK_THREADS 1024
#endif
static constexpr int kPkThreads = CUADMM_PK_THREADS;
static constexpr int kPkRecHeader = 8 + 32 + 16 + 16 + 16 + 64;
static constexpr int kPkMaxRowEntries = 768;
static constexpr int kPkMaxRows = 23000;
static constexpr int kPkChainMax = 384;        // unknowns in a collapsed chain (dense inverse kPkChainMax^2 / 2 entries)

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ long long pk_globaltimer() {
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

__device__ __forceinline__ void pk_fetch(unsigned char* dst, const unsigned char* src, uint64_t* bar) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(kPkChunk) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(smem_u32(dst)), "l"(src), "r"(kPkChunk), "r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ void pk_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                     : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    } while (!ok);
}

__device__ __forceinline__ void pk_record(const unsigned char* rec, int lane, double* xs) {
    // round 1: everything in the header is addressable from the lane id alone (a long record
    // replicates its single row into all 8 header positions)
    const int r = lane >> 2;
    const bool is_long = *reinterpret_cast<const int32_t*>(rec) != 0;
    const int ul = reinterpret_cast<const int32_t*>(rec + 8)[r];
    const int voff = reinterpret_cast<const uint16_t*>(rec + 40)[r];
    const int ioff = reinterpret_cast<const uint16_t*>(rec + 56)[r];
    const int ln = reinterpret_cast<const uint16_t*>(rec + 72)[r];
    const double invd = reinterpret_cast<const double*>(rec + 88)[r];
    const int j = is_long ? lane : (lane & 3);
    const int step = is_long ? 32 : 4;
    const double* val = reinterpret_cast<const double*>(rec) + voff;
    const uint16_t* idx = reinterpret_cast<const uint16_t*>(rec) + ioff;
    // round 2: values, indices, the slot's current content; round 3: the unknowns
    const double cur = ul >= 0 ? xs[ul] : 0.0;
    double acc = 0.0;
    for (int k = j; k < ln; k += step) acc = fma(val[k], xs[idx[k]], acc);
    acc += __shfl_xor_sync(0xffffffffu, acc, 1);
    acc += __shfl_xor_sync(0xffffffffu, acc, 2);
    if (is_long) {
        acc += __shfl_xor_sync(0xffffffffu, acc, 4);
        acc += __shfl_xor_sync(0xffffffffu, acc, 8);
        acc += __shfl_xor_sync(0xffffffffu, acc, 16);
    }
    if (ul >= 0 && j == 0) xs[ul] = (cur - acc) * invd;
}

// w[g] = rhs[src[g]] - sum over the row's dependencies OUTSIDE its subtree (all final by now) of
// val * x[dep], so the subtree kernels start from a coalesced read.  One thread per packed row in
// the first main_blocks CTAs; rows with many external entries (the collapsed chains at the top of
// a subtree touch hundreds of ancestors) are left to the remaining CTAs, one warp per row.
static constexpr int kPkHeavyExt = 8;

__global__ void __launch_bounds__(256) pk_gather_kernel(int64_t n_rows, int main_blocks, const int32_t* __restrict__ heavy,
        int n_heavy, const int32_t* __restrict__ prow_src, const int64_t* __restrict__ ext_ptr,
        const int32_t* __restrict__ ext_dep, const double* __restrict__ ext_val, const double* __restrict__ rhs,
        const double* __restrict__ x, double* __restrict__ w, const int* __restrict__ done_flag) {
    if (done_flag && *done_flag) return;
    if ((int)blockIdx.x < main_blocks) {
        const int64_t g = (int64_t)blockIdx.x * 256 + threadIdx.x;
        if (g >= n_rows) return;
        const int32_t src = prow_src[g];
        double acc = src >= 0 ? rhs[src] : 0.0;        // src < 0: a slot that starts from zero (see pack_subtrees)
        if (ext_ptr) {
            const int64_t p0 = ext_ptr[g], p1 = ext_ptr[g + 1];
            if (p1 - p0 > kPkHeavyExt) return;
            for (int64_t p = p0; p < p1; ++p) acc = fma(-ext_val[p], x[ext_dep[p]], acc);
        }
        w[g] = acc;
    } else {
        const int lane = threadIdx.x & 31;
        const int hw = ((int)blockIdx.x - main_blocks) * 8 + (threadIdx.x >> 5);
        if (hw >= n_heavy) return;
        const int64_t g = heavy[hw];
        double acc = 0.0;
        for (int64_t p = ext_ptr[g] + lane; p < ext_ptr[g + 1]; p += 32) acc = fma(ext_val[p], x[ext_dep[p]], acc);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) {
            const int32_t src = prow_src[g];
            w[g] = (src >= 0 ? rhs[src] : 0.0) - acc;
        }
    }
}

// Two records of one segment at a time (they are independent: same level).  A record is a chain of dependent
// shared-memory round trips (directory -> header -> value/index -> unknown -> shuffles), ~0.45 us for a warp that walks
// them one by one (measured: 1,729 records in 48 segments = 47 us for the largest subtree of the bench problem);
// interleaving two keeps twice as many loads in flight.  Every lane still adds its entries in the original order.
__device__ __forceinline__ void pk_record2(const unsigned char* recA, const unsigned char* recB, bool hasB, int lane, double* xs) {
    const int r = lane >> 2;
    const bool longA = *reinterpret_cast<const int32_t*>(recA) != 0;
    const bool longB = *reinterpret_cast<const int32_t*>(recB) != 0;
    const int ulA = reinterpret_cast<const int32_t*>(recA + 8)[r];
    const int ulB = hasB ? reinterpret_cast<const int32_t*>(recB + 8)[r] : -1;
    const int voffA = reinterpret_cast<const uint16_t*>(recA + 40)[r], voffB = reinterpret_cast<const uint16_t*>(recB + 40)[r];
    const int ioffA = reinterpret_cast<const uint16_t*>(recA + 56)[r], ioffB = reinterpret_cast<const uint16_t*>(recB + 56)[r];
    const int lnA = reinterpret_cast<const uint16_t*>(recA + 72)[r];
    const int lnB = hasB ? reinterpret_cast<const uint16_t*>(recB + 72)[r] : 0;
    const double invdA = reinterpret_cast<const double*>(recA + 88)[r], invdB = reinterpret_cast<const double*>(recB + 88)[r];
    const int jA = longA ? lane : (lane & 3), jB = longB ? lane : (lane & 3);
    const int stepA = longA ? 32 : 4, stepB = longB ? 32 : 4;
    const double* valA = reinterpret_cast<const double*>(recA) + voffA;
    const double* valB = reinterpret_cast<const double*>(recB) + voffB;
    const uint16_t* idxA = reinterpret_cast<const uint16_t*>(recA) + ioffA;
    const uint16_t* idxB = reinterpret_cast<const uint16_t*>(recB) + ioffB;
    const double curA = ulA >= 0 ? xs[ulA] : 0.0;
    const double curB = ulB >= 0 ? xs[ulB] : 0.0;
    double accA = 0.0, accB = 0.0;
    int kA = jA, kB = jB;
    while (kA < lnA || kB < lnB) {
        const bool a = kA < lnA, b = kB < lnB;
        double va = 0.0, vb = 0.0;
        int ia = 0, ib = 0;
        if (a) { va = valA[kA]; ia = idxA[kA]; }
        if (b) { vb = valB[kB]; ib = idxB[kB]; }
        const double xa = xs[ia], xb = xs[ib];
        if (a) accA = fma(va, xa, accA);
        if (b) accB = fma(vb, xb, accB);
        kA += stepA; kB += stepB;
    }
    accA += __shfl_xor_sync(0xffffffffu, accA, 1);
    accB += __shfl_xor_sync(0xffffffffu, accB, 1);
    accA += __shfl_xor_sync(0xffffffffu, accA, 2);
    accB += __shfl_xor_sync(0xffffffffu, accB, 2);
    if (longA || longB) {                       // warp-uniform; a short record's extra sums are discarded (only j == 0 stores)
        double tA = accA, tB = accB;
        tA += __shfl_xor_sync(0xffffffffu, tA, 4);  tB += __shfl_xor_sync(0xffffffffu, tB, 4);
        tA += __shfl_xor_sync(0xffffffffu, tA, 8);  tB += __shfl_xor_sync(0xffffffffu, tB, 8);
        tA += __shfl_xor_sync(0xffffffffu, tA, 16); tB += __shfl_xor_sync(0xffffffffu, tB, 16);
        if (longA) accA = tA;
        if (longB) accB = tB;
    }
    if (ulA >= 0 && jA == 0) xs[ulA] = (curA - accA) * invdA;
    if (ulB >= 0 && jB == 0) xs[ulB] = (curB - accB) * invdB;
}

// walk the segments of one chunk (resident in shared memory) with NW warps; WARP = the chunk belongs to one warp
template <int NW, bool WARP>
__device__ __forceinline__ void pk_chunk(const unsigned char* chunk, int lane, int warp, double* xs) {
    const uint16_t* dir = reinterpret_cast<const uint16_t*>(chunk);
    const int nseg = dir[0];
    const uint16_t* seg_end = dir + 2;
    const uint16_t* rec_off = seg_end + nseg;
    int sb = 0;
    for (int g = 0; g < nseg; ++g) {
        const int se = seg_end[g];
        int sl = sb + warp;
        if constexpr (!WARP) {      // (the one-warp subtrees have 1-2 records per level: pairing buys nothing there and costs registers)
            for (; sl + NW < se; sl += 2 * NW)
                pk_record2(chunk + 8 * (int)rec_off[sl], chunk + 8 * (int)rec_off[sl + NW], true, lane, xs);
        }
        for (; sl < se; sl += NW) pk_record(chunk + 8 * (int)rec_off[sl], lane, xs);
        if constexpr (WARP) __syncwarp(); else __syncthreads();
        sb = se;
    }
}

__global__ void __launch_bounds__(kPkThreads, 1) tri_packed_kernel(const int64_t* __restrict__ chunk_off,
        const int64_t* __restrict__ row_off, const unsigned char* __restrict__ stream, const int32_t* __restrict__ prow_u,
        const int32_t* __restrict__ prow_out, const double* __restrict__ w, double* x, double* out_scatter,
        const int* __restrict__ done_flag, long long* __restrict__ timeline) {
    if (done_flag && *done_flag) return;
    if (timeline && threadIdx.x == 0) timeline[4 * blockIdx.x + 0] = pk_globaltimer();
    extern __shared__ __align__(128) unsigned char pk_smem[];
    unsigned char* ring = pk_smem;
    uint64_t* bars = reinterpret_cast<uint64_t*>(pk_smem + kPkRing * kPkChunk);
    double* xs = reinterpret_cast<double*>(pk_smem + kPkRing * kPkChunk + 64);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t c0 = chunk_off[blockIdx.x];
    const int nc = (int)(chunk_off[blockIdx.x + 1] - c0);
    const int64_t r0 = row_off[blockIdx.x];
    const int nr = (int)(row_off[blockIdx.x + 1] - r0);
    const unsigned char* src = stream + c0 * kPkChunk;
    if (tid == 0) {
        for (int i = 0; i < kPkRing; ++i)
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(smem_u32(bars + i)) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        for (int i = 0; i < kPkRing && i < nc; ++i) pk_fetch(ring + i * kPkChunk, src + (int64_t)i * kPkChunk, bars + i);
    }
#pragma unroll 4
    for (int loc = tid; loc < nr; loc += kPkThreads) xs[loc] = w[r0 + loc];
    __syncthreads();     // xs ready, barriers initialised
    if (timeline && tid == 0) timeline[4 * blockIdx.x + 1] = pk_globaltimer();
    for (int c = 0; c < nc; ++c) {
        const int b = c % kPkRing;
        pk_wait(bars + b, (uint32_t)((c / kPkRing) & 1));
        pk_chunk<kPkThreads / 32, false>(ring + b * kPkChunk, lane, warp, xs);
        // every thread is past its last read of this ring buffer (a segment ends with a barrier): refill it
        if (tid == 0 && c + kPkRing < nc) pk_fetch(ring + b * kPkChunk, src + (int64_t)(c + kPkRing) * kPkChunk, bars + b);
    }
    if (timeline && tid == 0) timeline[4 * blockIdx.x + 2] = pk_globaltimer();
#pragma unroll 4
    for (int loc = tid; loc < nr; loc += kPkThreads) {
        const int32_t u = prow_u[r0 + loc];
        if (u < 0) continue;                        // scratch slot, not an unknown
        const double r = xs[loc];
        x[u] = r;
        if (out_scatter) out_scatter[prow_out[r0 + loc]] = r;
    }
    if (timeline && tid == 0) timeline[4 * blockIdx.x + 3] = pk_globaltimer();
}

// Tiny subtrees (tens of thousands of 2-8 row chains hanging off the spine of the elimination tree):
// one WARP per subtree.  Its whole packed description is one small blob (same format as a chunk),
// copied to the warp's slice of shared memory with coalesced 16-byte loads; the levels then run
// out of shared memory with __syncwarp: two global round trips per subtree instead of four per level.
static constexpr int kPkWarpBlob = 2048;      // bytes; bigger subtrees go to tri_packed_kernel
static constexpr int kPkWarpRows = 32;
static constexpr int kPkWarpThreads = 256;

__global__ void __launch_bounds__(kPkWarpThreads, 5) tri_packed_warp_kernel(int64_t count, const int64_t* __restrict__ blob_off,
        const int64_t* __restrict__ row_off, const uint4* __restrict__ blobs, const int32_t* __restrict__ prow_u,
        const int32_t* __restrict__ prow_out, const double* __restrict__ w, double* x, double* out_scatter,
        const int* __restrict__ done_flag) {
    if (done_flag && *done_flag) return;
    __shared__ __align__(16) unsigned char slices[kPkWarpThreads / 32][kPkWarpBlob];
    __shared__ double xs_all[kPkWarpThreads / 32][kPkWarpRows];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t t = (int64_t)blockIdx.x * (kPkWarpThreads / 32) + warp;
    if (t >= count) return;
    const int64_t b0 = blob_off[t];
    const int nb = (int)(blob_off[t + 1] - b0);          // 16-byte units
    const int64_t r0 = row_off[t];
    const int nr = (int)(row_off[t + 1] - r0);
    uint4* slice = reinterpret_cast<uint4*>(slices[warp]);
    double* xs = xs_all[warp];
    for (int i = lane; i < nb; i += 32) slice[i] = blobs[b0 + i];
    int32_t u = -1, po = -1;
    if (lane < nr) {
        xs[lane] = w[r0 + lane];
        u = prow_u[r0 + lane];
        if (out_scatter) po = prow_out[r0 + lane];
    }
    __syncwarp();
    pk_chunk<1, true>(slices[warp], lane, 0, xs);
    if (lane < nr && u >= 0) {
        const double r = xs[lane];
        x[u] = r;
        if (out_scatter) out_scatter[po] = r;
    }
}

// dense tail, single GPU: out[i] = sum_j T[i, j] * in[j] for an r x r triangular matrix (L22^-1 or its transpose) in
// tile-run storage (TailMatrix): per 64-row tile row, tile_ptr / tile_col list the runs of consecutive non-empty
// 64 x 64 tiles as [first, last) columns, and run t sits at T + tile_off[t], 64 rows of its full width.  Only those
// tiles are read.  One warp per row, coalesced 16-byte loads (run widths and offsets are multiples of 64 doubles).
// blk_order lists the 8-row blocks longest rows first, so the grid's tail wave is made of short rows.
__global__ void __launch_bounds__(256) tail_gemv_row_kernel(int64_t r, const double* __restrict__ T, const double* __restrict__ in,
                                                        double* out, const int32_t* __restrict__ tile_ptr,
                                                        const int32_t* __restrict__ tile_col, const int64_t* __restrict__ tile_off,
                                                        const int32_t* __restrict__ blk_order, double* out_scatter,
                                                        const int32_t* __restrict__ out_perm, int64_t perm_base,
                                                        const int* __restrict__ done_flag) {
    if (done_flag && *done_flag) return;
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blk_order[blockIdx.x] * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= r) return;
    const int I = (int)(row >> 6);
    double acc0 = 0.0, acc1 = 0.0;
    const bool in_al = (reinterpret_cast<uintptr_t>(in) & 15) == 0;
    for (int t = tile_ptr[I]; t < tile_ptr[I + 1]; ++t) {
        const int64_t j0 = tile_col[2 * t];
        const int64_t w = tile_col[2 * t + 1] - j0;
        const int64_t n = min(w, r - j0);                        // columns of the run inside the matrix
        const int64_t nv = n & ~(int64_t)1;
        const double* Ti = T + tile_off[t] + (row & 63) * w;
        const double* x = in + j0;
#pragma unroll 4      // measured: 8 or 16 loads in flight per lane are 7-8 % slower per solve (fewer resident warps)
        for (int64_t k = 2 * lane; k < nv; k += 64) {
            const double2 a = __ldcs(reinterpret_cast<const double2*>(Ti + k));   // streamed once: evict first
            const double2 b = in_al ? *reinterpret_cast<const double2*>(x + k) : make_double2(x[k], x[k + 1]);
            acc0 = fma(a.x, b.x, acc0);
            acc1 = fma(a.y, b.y, acc1);
        }
        if (lane == 0 && nv < n) acc0 = fma(Ti[nv], x[nv], acc0);
    }
    double acc = acc0 + acc1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) {
        out[row] = acc;
        if (out_scatter) out_scatter[out_perm[perm_base + row]] = acc;
    }
}

// Sharded solver (and any launch over a SUBSET of the rows): the row-per-warp kernel above is bound by the dependent load
// chain of its longest row (~30 us for 10k columns) however few rows it is given, so splitting rows over ranks buys
// nothing with it.  Here:
// One CTA = 8 consecutive rows x all their columns: warp w takes the 64-column chunks c == w (mod 8) of the tile row's
// runs for ALL 8 rows (8 independent accumulators, the input chunk loaded once for the 8 rows), then the 8 x 8 partials
// are reduced through shared memory.  A single row of 10k columns used to be one warp's dependent chain of ~160 loads
// (~30 us however few rows the launch had — which is why splitting the rows over ranks bought nothing); now the longest
// chain is 1/8 of that and every step has 9 loads in flight per lane.
// Sharded solver (npush > 0): this rank computes rows [row0, row0 + nrows) only and stores each result into every
// rank's copy of `out` over peer memory (one coalesced 64-byte store per CTA and peer); the kernel ends with the
// peer_leave handshake, so when it retires every rank holds the complete vector.  No peer_enter is needed: a peer
// can only reach this kernel after the handshake of the previous one, which this rank joined after its last read of
// the buffers.  row0 is a multiple of 8, so the 8 rows of a CTA share one 64-row tile row (= one list of column runs).
// Storage as in tail_gemv_row_kernel; blk_order lists this launch's 8-row blocks (from row0), longest rows first.
__global__ void __launch_bounds__(256) tail_gemv_kernel(int64_t r, const double* __restrict__ T, const double* in,
                                                        double* out, const int32_t* __restrict__ tile_ptr,
                                                        const int32_t* __restrict__ tile_col, const int64_t* __restrict__ tile_off,
                                                        const int32_t* __restrict__ blk_order, double* out_scatter,
                                                        const int32_t* __restrict__ out_perm, int64_t perm_base,
                                                        const int* __restrict__ done_flag,
                                                        int64_t row0, int64_t nrows, int npush, PeerView pv,
                                                        PeerPtrs outp, PeerPtrs scatp, int splits, double* split_part,
                                                        unsigned int* split_count) {
    if (done_flag && *done_flag) return;
    __shared__ double part[8][9];
    __shared__ int s_final;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    unsigned long long ep = 0;
    if (npush) ep = peer_epoch(pv);
    // `splits` CTAs share one block of 8 rows (groups of 8 consecutive chunks go round-robin over them): a rank's share of
    // the rows is too few CTAs to pull its share of the bytes at one CTA per row block (measured 20 us for 1/8 of the
    // rows).  The CTA that finds the other partials written adds them in split order (bit-identical on every rank).
    const int sp = (int)(blockIdx.x % (unsigned)splits);
    const int64_t rb = blockIdx.x / (unsigned)splits;
    const int64_t base = row0 + (int64_t)blk_order[rb] * 8;
    const int nr = (int)max((int64_t)0, min((int64_t)8, row0 + nrows - base));     // rows of this CTA
    double acc[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) acc[q] = 0.0;
    if (nr > 0) {
        const int I = (int)(base >> 6);
        const bool vec = (reinterpret_cast<uintptr_t>(in) & 15) == 0;   // run rows are 16-byte aligned
        int g = 0;                                        // running chunk index over the runs of this tile row
        for (int t = tile_ptr[I]; t < tile_ptr[I + 1]; ++t) {
            const int64_t j0 = tile_col[2 * t];
            const int64_t rw = tile_col[2 * t + 1] - j0;              // run width (row stride of the run)
            const int64_t n = min(rw, r - j0);                        // columns of the run inside the matrix
            const double* Tb = T + tile_off[t] + (base & 63) * rw;    // Tb[q * rw + k]: row base + q, column j0 + k
            const double* x = in + j0;
            const int nch = (int)((n + 63) >> 6);
            // chunk with running index G = g + c belongs to warp G & 7 of split (G >> 3) % splits
            const int g0 = g;
            int c = (w - (g & 7)) & 7;
            g += nch;
            for (; c < nch; c += 8) {
                if (splits > 1 && (((g0 + c) >> 3) % splits) != sp) continue;
                const int64_t k = ((int64_t)c << 6) + 2 * lane;
                if (vec) {
                    if (k + 1 < n) {
                        const double2 b = *reinterpret_cast<const double2*>(x + k);
#pragma unroll
                        for (int q = 0; q < 8; ++q) {
                            if (q < nr) {
                                const double2 a = __ldcs(reinterpret_cast<const double2*>(Tb + q * rw + k));   // streamed once
                                acc[q] = fma(a.x, b.x, fma(a.y, b.y, acc[q]));
                            }
                        }
                    } else if (k < n) {
                        const double b = x[k];
#pragma unroll
                        for (int q = 0; q < 8; ++q) if (q < nr) acc[q] = fma(Tb[q * rw + k], b, acc[q]);
                    }
                } else {
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const int64_t kk = ((int64_t)c << 6) + lane + 32 * h;
                        if (kk < n) {
                            const double b = x[kk];
#pragma unroll
                            for (int q = 0; q < 8; ++q) if (q < nr) acc[q] = fma(Tb[q * rw + kk], b, acc[q]);
                        }
                    }
                }
            }
        }
    }
#pragma unroll
    for (int q = 0; q < 8; ++q) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc[q] += __shfl_xor_sync(0xffffffffu, acc[q], o);
    }
    if (lane == 0) {
#pragma unroll
        for (int q = 0; q < 8; ++q) part[w][q] = acc[q];
    }
    __syncthreads();
    const int t = threadIdx.x;
    bool final_cta = true;
    if (splits > 1) {
        if (t < 8) {
            double v = 0.0;
#pragma unroll
            for (int k = 0; k < 8; ++k) v += part[k][t];
            split_part[(rb * splits + sp) * 8 + t] = v;
        }
        __syncthreads();
        if (t == 0) {
            __threadfence();
            const unsigned old = atomicAdd(split_count + rb, 1u);
            s_final = (old == (unsigned)splits - 1u) ? 1 : 0;
            if (s_final) { split_count[rb] = 0u; __threadfence(); }
        }
        __syncthreads();
        final_cta = s_final != 0;
    }
    if (final_cta && t < 8 * max(npush, 1)) {
        const int q = t >> 3, rr = t & 7;
        if (rr < nr) {
            double v = 0.0;
            if (splits > 1) {
                for (int k = 0; k < splits; ++k) v += __ldcg(split_part + (rb * splits + k) * 8 + rr);   // split order
            } else {
#pragma unroll
                for (int k = 0; k < 8; ++k) v += part[k][rr];      // fixed order: identical on every rank
            }
            if (npush == 0) {
                out[base + rr] = v;
                if (out_scatter) out_scatter[out_perm[perm_base + base + rr]] = v;
            } else {
                outp.p[q][base + rr] = v;
            }
        }
    }
    if (npush) peer_leave(pv, ep);
}

// y[perm[base + i]] = x_tail[i]: the scatter of the dense-tail solution into y (sharded solver; local)
__global__ void __launch_bounds__(256) tail_scatter_kernel(int64_t r, const double* __restrict__ xt, const int32_t* __restrict__ perm,
                                                           int64_t base, double* y, const int* __restrict__ done_flag) {
    if (done_flag && *done_flag) return;
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i < r) y[perm[base + i]] = xt[i];
}

// gather/external fold, then the packed CTA-per-subtree kernel on `st` and the warp-per-subtree kernel
// concurrently on `side` (fork/join by events); the generic kernel only for subtrees that cannot be packed
static int launch_subtrees(const TriSweep& S, const double* rhs, const int32_t* gather, double* x, double* out_scatter,
                           const int32_t* out_perm, const int* done, cudaStream_t st, const SweepStreams& ss) {
    int launches = 0;
    if (S.pk_rows > 0) {
        const int main_blocks = (int)((S.pk_rows + 255) / 256);
        pk_gather_kernel<<<(unsigned)(main_blocks + (S.pk_n_heavy + 7) / 8), 256, 0, st>>>(S.pk_rows, main_blocks, S.pk_heavy.p,
            (int)S.pk_n_heavy, S.pk_prow_src.p, S.pk_has_ext ? S.pk_ext_ptr.p : nullptr, S.pk_ext_dep.p, S.pk_ext_val.p, rhs, x,
            S.pk_w.p, done);
        ++launches;
    }
    const bool fork = S.n_sub_warp > 0 && (S.n_sub_pack > 0 || S.n_sub_cta > 0);
    cudaStream_t wst = st;
    if (fork) {
        CUADMM_CUDA(cudaEventRecord(ss.fork, st));
        CUADMM_CUDA(cudaStreamWaitEvent(ss.side, ss.fork, 0));
        wst = ss.side;
    }
    if (S.n_sub_pack > 0) {
        tri_packed_kernel<<<(unsigned)S.n_sub_pack, kPkThreads, S.pk_smem, st>>>(S.pk_chunk_off.p, S.pk_row_off.p, S.pk_stream.p,
            S.pk_prow_u.p, S.pk_prow_out.p, S.pk_w.p, x, out_scatter, done, S.pk_timeline.n ? S.pk_timeline.p : nullptr);
        ++launches;
    }
    if (S.n_sub_warp > 0) {
        const int wpb = kPkWarpThreads / 32;
        tri_packed_warp_kernel<<<(unsigned)((S.n_sub_warp + wpb - 1) / wpb), kPkWarpThreads, 0, wst>>>(S.n_sub_warp,
            S.pk_blob_off.p, S.pk_row_off.p + S.n_sub_pack, reinterpret_cast<const uint4*>(S.pk_blobs.p), S.pk_prow_u.p,
            S.pk_prow_out.p, S.pk_w.p, x, out_scatter, done);
        ++launches;
    }
    if (S.n_sub_cta > 0) {
        tri_subtree_kernel<<<(unsigned)S.n_sub_cta, kTriThreads, 0, st>>>(S.sub_off.p, S.sub_lvl_ptr.p, S.slot_rows.p, S.slot_info.p,
            S.ptr.p, S.dep.p, S.val.p, S.inv_diag.p, rhs, gather, x, out_scatter, out_perm, done);
        ++launches;
    }
    if (fork) {
        CUADMM_CUDA(cudaEventRecord(ss.join, ss.side));
        CUADMM_CUDA(cudaStreamWaitEvent(st, ss.join, 0));
    }
    return launches;
}

static int launch_sweep(const TriSweep& S, const double* rhs, const int32_t* gather, double* x,
                        double* out_scatter, const int32_t* out_perm, const int* done, cudaStream_t st, const SweepStreams& ss) {
    int launches = 0;
    if (S.subtrees_first && S.n_sub) launches += launch_subtrees(S, rhs, gather, x, out_scatter, out_perm, done, st, ss);
    for (const TriSweep::Phase& ph : S.phases) {
        if (ph.narrow) {
            tri_narrow_kernel<<<1, kNarrowThreads, 0, st>>>(ph.level0, ph.level1, S.level_ptr.p, S.slot_rows.p, S.slot_info.p,
                S.ptr.p, S.dep.p, S.val.p, S.inv_diag.p, rhs, gather, x, out_scatter, out_perm, done);
        } else {
            const int64_t s0 = S.h_level_ptr[ph.level0], s1 = S.h_level_ptr[ph.level1];
            const int grid = (int)(((s1 - s0) * 32 + kTriThreads - 1) / kTriThreads);
            tri_wide_kernel<<<grid, kTriThreads, 0, st>>>(s0, s1, S.slot_rows.p, S.slot_info.p, S.ptr.p, S.dep.p, S.val.p,
                S.inv_diag.p, rhs, gather, x, out_scatter, out_perm, done);
        }
        ++launches;
    }
    if (!S.subtrees_first && S.n_sub) launches += launch_subtrees(S, rhs, gather, x, out_scatter, out_perm, done, st, ss);
    CUADMM_CUDA(cudaGetLastError());
    return launches;
}

// host: pull structure -> device sweep
struct HostSweep {
    std::vector<int64_t> ptr;
    std::vector<int32_t> dep;
    std::vector<double> val, inv_diag;
    int64_t n = 0;                  // unknown id space
    std::vector<int32_t> order;     // the unknowns of this sweep in a valid (topological) solve order
    std::vector<int32_t> sub;       // per unknown id: subtree id, or -1 = top part
    int64_t n_sub = 0;
    bool subtrees_first = true;     // forward: subtrees then top; backward: top then subtrees
    const std::vector<int32_t>* gather = nullptr;     // rhs is read at gather[u] (null: at u)
    const std::vector<int32_t>* out_perm = nullptr;   // results are also scattered to out[out_perm[u]] (null: no scatter)
};

// slots for a list of unknowns that all belong to one level
static int64_t emit_level_slots(const HostSweep& H, std::vector<int32_t>& rows, int level,
                                std::vector<int32_t>& slot_rows, std::vector<int32_t>& slot_info) {
    std::vector<int32_t> longs, shorts;
    for (int32_t u : rows) ((H.ptr[u + 1] - H.ptr[u]) > kLongRowNnz ? longs : shorts).push_back(u);
    std::stable_sort(longs.begin(), longs.end(), [&](int32_t a, int32_t b) {
        return H.ptr[a + 1] - H.ptr[a] > H.ptr[b + 1] - H.ptr[b]; });
    int64_t cnt = 0;
    for (int32_t u : longs) {
        slot_rows.push_back(u);
        for (int t = 1; t < 8; ++t) slot_rows.push_back(-1);
        slot_info.push_back(level | (1 << 30));
        ++cnt;
    }
    for (size_t t = 0; t < shorts.size(); t += 8) {
        for (size_t q = t; q < t + 8; ++q) slot_rows.push_back(q < shorts.size() ? shorts[q] : -1);
        slot_info.push_back(level);
        ++cnt;
    }
    return cnt;
}

// Host side of the packed subtree kernels.  Decides per subtree: 2 = CTA-packed (chunk stream),
// 1 = warp-packed (one small blob), 0 = not packable (generic kernel); builds the streams, the unified
// slot lists (CTA-packed subtrees first, then warp-packed) and the external (out-of-subtree) entries.
//
// Chain collapse.  The top of a subtree of the elimination tree is typically a chain: ~130 levels of
// ONE dense-ish row each, i.e. a small dense triangular system L_CC solved one row per barrier.  For
// such a set C (at most kPkChainMax unknowns, chosen by level so that it is closed the right way) the
// host inverts L_CC once, M = L_CC^-1, and the sweep computes x_C = M t_C as ONE level of independent
// dense rows, t_C = b_C - (contributions from outside C).  Two flavours, whichever the sweep needs:
//   final set   (forward sweep):  C = {level >= l0}; nothing outside C depends on C;
//                                 levels: R rows (unchanged), t_C = b_C - L_CR x_R, x_C = M t_C;
//   initial set (backward sweep): C = {height >= h0}; C depends on nothing outside C (in the subtree);
//                                 levels: x_C = M t_C, then the R rows with levels counted inside R.
// t_C lives in extra scratch slots behind the subtree's unknowns so that x_C = M t_C has no in-place hazard.
struct PkRow {                       // one row of one level: slot = (slot - sum val * xs[idx]) * invd
    int32_t slot; double invd;
    std::vector<uint16_t> idx; std::vector<double> val;
};

static void pack_subtrees(const HostSweep& H, TriSweep& S, const std::vector<std::vector<int32_t>>& members,
                          const std::vector<int32_t>& level, const std::vector<int32_t>& depth, std::vector<int>& kind) {
    struct Packed {
        std::vector<unsigned char> bytes; int32_t t; size_t last_used; int levels;
        std::vector<int32_t> slot_u, slot_src;      // per slot: unknown to write (-1 none), unknown to start from (-1: zero)
    };
    std::vector<Packed> packs, blobs;
    std::vector<int32_t> loc(H.n, -1), cidx(H.n, -1), height(H.n, 0), lvl_r(H.n, 0);
    int chain_max = kPkChainMax, chain_gain = 6;
    if (const char* e = getenv("CUADMM_SWEEP_CHAIN_MAX")) chain_max = std::min(atoi(e), kPkMaxRowEntries);
    const bool verbose = getenv("CUADMM_YSOLVE_VERBOSE") != nullptr;
    int64_t n_collapsed = 0, levels_before = 0, levels_after = 0, chain_entries = 0;
    kind.assign(H.n_sub, 0);
    auto same = [&](int32_t u, int64_t p) { return H.sub[H.dep[p]] == H.sub[u]; };
    // one subtree at a time, on a pool of host threads: subtrees own disjoint rows of the scratch arrays (loc, cidx, height,
    // lvl_r), results land in per-subtree slots and are collected in subtree order afterwards (deterministic layout)
    std::vector<Packed> result(H.n_sub);
    std::atomic<int64_t> a_collapsed{0}, a_before{0}, a_after{0}, a_entries{0};
    auto do_subtree = [&](int64_t t) {
        const std::vector<int32_t>& rows = members[t];       // in solve order
        const int32_t nr0 = (int32_t)rows.size();
        if (nr0 + chain_max > kPkMaxRows) return;
        int32_t longest = 0;
        for (int32_t q = 0; q < nr0; ++q) {
            const int32_t u = rows[q];
            loc[u] = q;
            int32_t cnt = 0;
            for (int64_t p = H.ptr[u]; p < H.ptr[u + 1]; ++p) cnt += same(u, p) ? 1 : 0;
            longest = std::max(longest, cnt);
        }
        if (longest > kPkMaxRowEntries) return;
        // ---- chain collapse: pick C
        std::vector<int32_t> C;
        int new_depth = depth[t], k0 = 0;
        if (chain_max > 0 && depth[t] > chain_gain + 2 && nr0 > kPkWarpRows) {
            const bool initial = !H.subtrees_first;             // backward sweep
            std::vector<int32_t> key(nr0);
            if (initial) {
                for (int32_t u : rows) height[u] = 0;
                for (int32_t q = nr0 - 1; q >= 0; --q) {        // reverse solve order: dependents first
                    const int32_t u = rows[q];
                    for (int64_t p = H.ptr[u]; p < H.ptr[u + 1]; ++p)
                        if (same(u, p)) height[H.dep[p]] = std::max(height[H.dep[p]], height[u] + 1);
                }
                for (int32_t q = 0; q < nr0; ++q) key[q] = height[rows[q]];
            } else {
                for (int32_t q = 0; q < nr0; ++q) key[q] = level[rows[q]];
            }
            std::vector<int32_t> cnt(depth[t] + 1, 0);
            for (int32_t q = 0; q < nr0; ++q) ++cnt[key[q]];
            int32_t acc = 0;
            k0 = depth[t];
            while (k0 > 0 && acc + cnt[k0 - 1] <= chain_max) { --k0; acc += cnt[k0]; }
            const int nd = initial ? k0 + 1 : k0 + 2;
            if (acc > 0 && depth[t] - nd >= chain_gain) {
                new_depth = nd;
                for (int32_t q = 0; q < nr0; ++q) if (key[q] >= k0) C.push_back(rows[q]);   // solve order = topological
            }
        }
        const int32_t nC = (int32_t)C.size();
        for (int32_t i = 0; i < nC; ++i) cidx[C[i]] = i;
        // ---- levels of PkRow
        std::vector<std::vector<PkRow>> lv(new_depth);
        auto plain_row = [&](int32_t u) {
            PkRow r; r.slot = loc[u]; r.invd = H.inv_diag[u];
            for (int64_t p = H.ptr[u]; p < H.ptr[u + 1]; ++p)
                if (same(u, p)) { r.idx.push_back((uint16_t)loc[H.dep[p]]); r.val.push_back(H.val[p]); }
            return r;
        };
        if (nC == 0) {
            for (int32_t u : rows) lv[level[u]].push_back(plain_row(u));
        } else {
            // M = L_CC^-1 by rows:  M[c,:] = invd_c * (e_c - sum_{k in C} v_ck M[k,:])
            std::vector<double> M((size_t)nC * nC, 0.0);
            for (int32_t i = 0; i < nC; ++i) {
                const int32_t u = C[i];
                double* mi = M.data() + (size_t)i * nC;
                mi[i] = 1.0;
                for (int64_t p = H.ptr[u]; p < H.ptr[u + 1]; ++p) {
                    if (!same(u, p) || cidx[H.dep[p]] < 0) continue;
                    const int32_t k = cidx[H.dep[p]];
                    const double v = H.val[p];
                    const double* mk = M.data() + (size_t)k * nC;
                    for (int32_t j = 0; j <= k; ++j) mi[j] -= v * mk[j];
                }
                const double d = H.inv_diag[u];
                for (int32_t j = 0; j <= i; ++j) mi[j] *= d;
            }
            const bool initial = !H.subtrees_first;
            const int lvB = initial ? 0 : k0 + 1;
            for (int32_t i = 0; i < nC; ++i) {          // x_C = M t_C:  x = (0 - sum M t) * (-1)
                PkRow r; r.slot = loc[C[i]]; r.invd = -1.0;
                const double* mi = M.data() + (size_t)i * nC;
                for (int32_t j = 0; j <= i; ++j) if (mi[j] != 0.0) { r.idx.push_back((uint16_t)(nr0 + j)); r.val.push_back(mi[j]); }
                a_entries += (int64_t)r.idx.size();
                lv[lvB].push_back(std::move(r));
            }
            if (initial) {
                for (int32_t u : rows) {
                    if (cidx[u] >= 0) continue;
                    int32_t l = 0;
                    for (int64_t p = H.ptr[u]; p < H.ptr[u + 1]; ++p)
                        if (same(u, p) && cidx[H.dep[p]] < 0) l = std::max(l, lvl_r[H.dep[p]] + 1);
                    lvl_r[u] = l;
                    lv[1 + l].push_back(plain_row(u));
                }
            } else {
                for (int32_t u : rows) {
                    if (cidx[u] < 0) { lv[level[u]].push_back(plain_row(u)); continue; }
                    PkRow r; r.slot = nr0 + cidx[u]; r.invd = 1.0;     // t_c = b_c - L_cR x_R
                    for (int64_t p = H.ptr[u]; p < H.ptr[u + 1]; ++p)
                        if (same(u, p) && cidx[H.dep[p]] < 0) { r.idx.push_back((uint16_t)loc[H.dep[p]]); r.val.push_back(H.val[p]); }
                    if (!r.idx.empty()) lv[k0].push_back(std::move(r));
                }
            }
            ++a_collapsed; a_before += depth[t]; a_after += new_depth;
        }
        // ---- records and chunks
        Packed& P = result[t]; P.t = (int32_t)t; P.last_used = 0; P.levels = new_depth;
        P.slot_u.assign(nr0 + nC, -1); P.slot_src.assign(nr0 + nC, -1);
        for (int32_t q = 0; q < nr0; ++q) {
            const int32_t u = rows[q];
            P.slot_u[q] = u;
            if (cidx[u] < 0) P.slot_src[q] = u; else P.slot_src[nr0 + cidx[u]] = u;
        }
        std::vector<uint16_t> seg_end, rec_rel;      // open chunk; rec_rel: record offsets (bytes) inside the records area
        std::vector<unsigned char> recs;
        auto dir_bytes = [](size_t nseg, size_t nslots) { return (4 + 2 * nseg + 2 * nslots + 7) / 8 * 8; };
        auto close_chunk = [&]() {
            if (rec_rel.empty()) return;
            seg_end.push_back((uint16_t)rec_rel.size());
            const size_t db = dir_bytes(seg_end.size(), rec_rel.size());
            // a chunk is stored unpadded until another one follows it (tens of thousands of tiny subtrees have one short
            // chunk each: padding every one to kPkChunk zero-filled gigabytes at init)
            if (!P.bytes.empty()) P.bytes.resize((P.bytes.size() + kPkChunk - 1) / kPkChunk * kPkChunk, 0);
            std::vector<unsigned char> chunk((db + recs.size() + 15) / 16 * 16, 0);
            uint16_t* dir = reinterpret_cast<uint16_t*>(chunk.data());
            dir[0] = (uint16_t)seg_end.size(); dir[1] = (uint16_t)rec_rel.size();
            for (size_t i = 0; i < seg_end.size(); ++i) dir[2 + i] = seg_end[i];
            for (size_t i = 0; i < rec_rel.size(); ++i) dir[2 + seg_end.size() + i] = (uint16_t)((db + rec_rel[i]) / 8);
            CUADMM_REQUIRE(db + recs.size() <= (size_t)kPkChunk, "internal: packed chunk overflow");
            std::copy(recs.begin(), recs.end(), chunk.begin() + db);
            P.bytes.insert(P.bytes.end(), chunk.begin(), chunk.end());
            P.last_used = db + recs.size();
            seg_end.clear(); rec_rel.clear(); recs.clear();
        };
        auto add_record = [&](const std::vector<unsigned char>& rec, bool new_level) {
            const size_t nseg = seg_end.size() + 1 + ((new_level && !rec_rel.empty()) ? 1 : 0);
            if (dir_bytes(nseg, rec_rel.size() + 1) + recs.size() + rec.size() > (size_t)kPkChunk) close_chunk();
            if (new_level && !rec_rel.empty()) seg_end.push_back((uint16_t)rec_rel.size());
            rec_rel.push_back((uint16_t)recs.size());
            recs.insert(recs.end(), rec.begin(), rec.end());
        };
        auto make_record = [&](const PkRow* const* rs, int nrows, bool is_long) {
            size_t ne = 0;
            for (int r = 0; r < nrows; ++r) ne += rs[r]->val.size();
            const size_t val0 = kPkRecHeader, idx0 = kPkRecHeader + 8 * ne;
            std::vector<unsigned char> rec(idx0 + (2 * ne + 7) / 8 * 8, 0);
            int32_t* hdr = reinterpret_cast<int32_t*>(rec.data());
            int32_t* slot = hdr + 2;
            uint16_t* voff = reinterpret_cast<uint16_t*>(rec.data() + 40);
            uint16_t* ioff = reinterpret_cast<uint16_t*>(rec.data() + 56);
            uint16_t* len = reinterpret_cast<uint16_t*>(rec.data() + 72);
            double* invd = reinterpret_cast<double*>(rec.data() + 88);
            double* val = reinterpret_cast<double*>(rec.data() + val0);
            uint16_t* idx = reinterpret_cast<uint16_t*>(rec.data() + idx0);
            hdr[0] = is_long ? 1 : 0; hdr[1] = (int32_t)ne;
            size_t e = 0;
            for (int r = 0; r < 8; ++r) {
                slot[r] = -1; voff[r] = (uint16_t)(val0 / 8); ioff[r] = (uint16_t)(idx0 / 2); len[r] = 0; invd[r] = 0.0;
                const PkRow* row = is_long ? rs[0] : (r < nrows ? rs[r] : nullptr);
                if (!row) continue;
                if (is_long && r > 0) {        // replicate row 0
                    slot[r] = slot[0]; voff[r] = voff[0]; ioff[r] = ioff[0]; len[r] = len[0]; invd[r] = invd[0];
                    continue;
                }
                slot[r] = row->slot; invd[r] = row->invd; len[r] = (uint16_t)row->val.size();
                voff[r] = (uint16_t)((val0 + 8 * e) / 8); ioff[r] = (uint16_t)((idx0 + 2 * e) / 2);
                std::copy(row->val.begin(), row->val.end(), val + e);
                std::copy(row->idx.begin(), row->idx.end(), idx + e);
                e += row->val.size();
            }
            return rec;
        };
        for (int l = 0; l < new_depth; ++l) {
            std::vector<const PkRow*> longs, shorts;
            for (const PkRow& r : lv[l]) ((int)r.idx.size() > kLongRowNnz ? longs : shorts).push_back(&r);
            if (nr0 > kPkWarpRows && !shorts.empty()) {
                // CTA subtree, thin level (fewer records than the 32 warps of the CTA): its time is the longest row's chain
                // of dependent index -> unknown loads, 4 lanes per row = up to 6 rounds.  Warps are idle anyway, so the
                // longest rows get a whole warp each (one round) as long as every record still has its own warp.
                constexpr int kWarps = kPkThreads / 32;
                std::stable_sort(shorts.begin(), shorts.end(), [](const PkRow* a, const PkRow* b) { return a->idx.size() > b->idx.size(); });
                size_t promote = 0;
                while (promote < shorts.size() && shorts[promote]->idx.size() > 4 &&
                       longs.size() + promote + 1 + (shorts.size() - promote - 1 + 7) / 8 <= (size_t)kWarps) ++promote;
                longs.insert(longs.end(), shorts.begin(), shorts.begin() + promote);
                shorts.erase(shorts.begin(), shorts.begin() + promote);
            }
            std::stable_sort(longs.begin(), longs.end(), [](const PkRow* a, const PkRow* b) { return a->idx.size() > b->idx.size(); });
            bool first = true;
            for (const PkRow* r : longs) { add_record(make_record(&r, 1, true), first); first = false; }
            for (size_t q = 0; q < shorts.size(); q += 8) {
                add_record(make_record(shorts.data() + q, (int)std::min<size_t>(8, shorts.size() - q), false), first);
                first = false;
            }
        }
        close_chunk();
        for (int32_t u : C) cidx[u] = -1;
        if (nC == 0 && nr0 <= kPkWarpRows && P.bytes.size() <= (size_t)kPkChunk && P.last_used <= (size_t)kPkWarpBlob) {
            P.bytes.resize((P.last_used + 15) / 16 * 16);
            kind[t] = 1;
        } else {
            kind[t] = 2;
        }
    };
    if (H.n_sub > 0) {
        int nthreads = (int)std::min<int64_t>(std::max(1u, std::thread::hardware_concurrency()), 32);
        if (const char* e = getenv("CUADMM_INIT_THREADS")) nthreads = std::max(1, atoi(e));
        nthreads = (int)std::min<int64_t>(nthreads, H.n_sub);
        std::atomic<int64_t> next{0};
        std::vector<std::string> errors(nthreads);
        auto worker = [&](int id) {
            try {
                for (int64_t t = next.fetch_add(1); t < H.n_sub; t = next.fetch_add(1)) do_subtree(t);
            } catch (const std::exception& ex) { errors[id] = ex.what(); next.store(H.n_sub); }
        };
        std::vector<std::thread> pool;
        for (int i = 1; i < nthreads; ++i) pool.emplace_back(worker, i);
        worker(0);
        for (auto& th : pool) th.join();
        for (const std::string& e : errors) if (!e.empty()) throw Error(CUADMM_EINVAL, e);
        for (int64_t t = 0; t < H.n_sub; ++t) {
            if (kind[t] == 1) blobs.push_back(std::move(result[t]));
            else if (kind[t] == 2) packs.push_back(std::move(result[t]));
        }
    }
    n_collapsed = a_collapsed; levels_before = a_before; levels_after = a_after; chain_entries = a_entries;
    S.n_sub_pack = (int64_t)packs.size();
    S.n_sub_warp = (int64_t)blobs.size();
    S.pk_smem = 0; S.pk_rows = 0;
    if (packs.empty() && blobs.empty()) return;
    // biggest first: CTAs are dispatched in index order
    std::stable_sort(packs.begin(), packs.end(), [](const Packed& a, const Packed& b) { return a.bytes.size() > b.bytes.size(); });
    std::stable_sort(blobs.begin(), blobs.end(), [&](const Packed& a, const Packed& b) { return a.levels > b.levels; });
    std::vector<int64_t> chunk_off(1, 0), blob_off(1, 0), row_off(1, 0), ext_ptr(1, 0);
    std::vector<int32_t> prow_u, prow_src, prow_out, ext_dep;
    std::vector<double> ext_val;
    std::vector<unsigned char> stream, blob_bytes;
    int64_t max_slots = 0;
    auto add_slots = [&](const Packed& P) {
        for (size_t q = 0; q < P.slot_u.size(); ++q) {
            const int32_t u = P.slot_u[q], su = P.slot_src[q];
            prow_u.push_back(u);
            prow_out.push_back((u >= 0 && H.out_perm) ? (*H.out_perm)[u] : 0);
            prow_src.push_back(su < 0 ? -1 : (H.gather ? (*H.gather)[su] : su));
            if (su >= 0)
                for (int64_t p = H.ptr[su]; p < H.ptr[su + 1]; ++p)
                    if (!same(su, p)) { ext_dep.push_back(H.dep[p]); ext_val.push_back(H.val[p]); }
            ext_ptr.push_back((int64_t)ext_dep.size());
        }
        row_off.push_back((int64_t)prow_u.size());
        max_slots = std::max<int64_t>(max_slots, (int64_t)P.slot_u.size());
    };
    for (const Packed& P : packs) {
        stream.insert(stream.end(), P.bytes.begin(), P.bytes.end());
        stream.resize((stream.size() + kPkChunk - 1) / kPkChunk * kPkChunk, 0);      // the last chunk of a pack is stored unpadded
        chunk_off.push_back((int64_t)(stream.size() / kPkChunk));
        add_slots(P);
    }
    const int64_t cta_slots = max_slots;
    for (const Packed& P : blobs) {
        blob_bytes.insert(blob_bytes.end(), P.bytes.begin(), P.bytes.end());
        blob_off.push_back((int64_t)(blob_bytes.size() / 16));
        add_slots(P);
    }
    S.pk_rows = (int64_t)prow_u.size();
    S.pk_has_ext = !ext_dep.empty();
    if (ext_dep.empty()) { ext_dep.push_back(0); ext_val.push_back(0.0); }
    if (stream.empty()) stream.assign(16, 0);
    if (blob_bytes.empty()) blob_bytes.assign(16, 0);
    S.pk_stream.upload(stream); S.pk_chunk_off.upload(chunk_off); S.pk_blobs.upload(blob_bytes); S.pk_blob_off.upload(blob_off);
    S.pk_row_off.upload(row_off); S.pk_prow_u.upload(prow_u); S.pk_prow_src.upload(prow_src); S.pk_prow_out.upload(prow_out);
    S.pk_ext_ptr.upload(ext_ptr); S.pk_ext_dep.upload(ext_dep); S.pk_ext_val.upload(ext_val);
    S.pk_w.alloc(S.pk_rows);
    std::vector<int32_t> heavy;
    for (int64_t g = 0; g < S.pk_rows; ++g) if (ext_ptr[g + 1] - ext_ptr[g] > kPkHeavyExt) heavy.push_back((int32_t)g);
    S.pk_n_heavy = (int64_t)heavy.size();
    if (heavy.empty()) heavy.push_back(0);
    S.pk_heavy.upload(heavy);
    if (getenv("CUADMM_YSOLVE_TIMELINE") && !packs.empty()) {   // debug: per-CTA globaltimer stamps of tri_packed_kernel
        S.pk_timeline.alloc(4 * (int64_t)packs.size());
        std::vector<long long> meta;
        for (const Packed& P : packs) { meta.push_back((long long)((P.bytes.size() + kPkChunk - 1) / kPkChunk)); meta.push_back((long long)P.slot_u.size()); meta.push_back(P.levels); }
        S.pk_timeline_meta = meta;
    }
    S.pk_smem = (size_t)kPkRing * kPkChunk + 64 + sizeof(double) * (size_t)cta_slots;
    CUADMM_CUDA(cudaFuncSetAttribute((const void*)tri_packed_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S.pk_smem));
    if (verbose)
        fprintf(stderr, "[ysolve] %s packed: %zu CTA subtrees in %lld chunks (largest %zu), %zu warp subtrees in %zu bytes, "
                "%lld slots, %lld external entries (%lld heavy rows), smem %zu; chains collapsed in %lld subtrees (%lld -> %lld levels, %lld inverse entries)\n",
                H.subtrees_first ? "fwd" : "bwd", packs.size(), (long long)chunk_off.back(),
                packs.empty() ? (size_t)0 : (packs[0].bytes.size() + kPkChunk - 1) / kPkChunk, blobs.size(), blob_bytes.size(), (long long)S.pk_rows,
                (long long)ext_ptr.back(), (long long)S.pk_n_heavy, S.pk_smem, (long long)n_collapsed, (long long)levels_before, (long long)levels_after,
                (long long)chain_entries);
}

static void upload_sweep(const HostSweep& H, TriSweep& S) {
    S.n_unknowns = (int64_t)H.order.size();
    S.nnz = (int64_t)H.dep.size();
    S.subtrees_first = H.subtrees_first;
    // levels inside each part (a subtree, or the top): dependencies that live in another part are
    // final by construction of the launch order and do not count
    std::vector<int32_t> level(H.n, 0);
    for (int32_t u : H.order) {
        int32_t l = 0;
        for (int64_t p = H.ptr[u]; p < H.ptr[u + 1]; ++p) {
            const int32_t d = H.dep[p];
            if (H.sub[d] == H.sub[u]) l = std::max(l, level[d] + 1);
        }
        level[u] = l;
    }
    std::vector<int32_t> slot_rows, slot_info;
    // ---- subtree part
    std::vector<std::vector<int32_t>> members(H.n_sub);
    std::vector<int32_t> depth(H.n_sub, 0);
    for (int32_t u : H.order) if (H.sub[u] >= 0) {
        members[H.sub[u]].push_back(u);
        depth[H.sub[u]] = std::max(depth[H.sub[u]], level[u] + 1);
    }
    std::vector<int> kind;
    pack_subtrees(H, S, members, level, depth, kind);
    // whatever could not be packed: generic CTA-per-subtree kernel, slots grouped by (subtree, level), deepest first
    std::vector<int32_t> sub_order;
    for (int64_t t = 0; t < H.n_sub; ++t) if (kind[t] == 0) sub_order.push_back((int32_t)t);
    std::stable_sort(sub_order.begin(), sub_order.end(), [&](int32_t a, int32_t b) { return depth[a] > depth[b]; });
    S.n_sub_cta = (int64_t)sub_order.size();
    std::vector<int64_t> sub_off(1, 0), sub_lvl_ptr;
    int max_sub_depth = 0;
    for (int32_t t : sub_order) {
        std::vector<std::vector<int32_t>> by_level(depth[t]);
        for (int32_t u : members[t]) by_level[level[u]].push_back(u);
        for (int l = 0; l < depth[t]; ++l) {
            sub_lvl_ptr.push_back((int64_t)slot_info.size());
            emit_level_slots(H, by_level[l], l, slot_rows, slot_info);
        }
        sub_lvl_ptr.push_back((int64_t)slot_info.size());
        sub_off.push_back((int64_t)sub_lvl_ptr.size());
    }
    for (int64_t t = 0; t < H.n_sub; ++t) max_sub_depth = std::max(max_sub_depth, depth[t]);
    S.n_sub = H.n_sub;
    S.sub_depth = max_sub_depth;
    if (getenv("CUADMM_YSOLVE_VERBOSE")) {
        const int64_t edges[] = {8, 32, 128, 256, 512, 1024, 2048, 4096, 1 << 30};
        for (int b = 0; b < 9; ++b) {
            int64_t cnt = 0, r = 0, dsum = 0; int dmax = 0;
            for (int64_t t = 0; t < H.n_sub; ++t) {
                const int64_t sz = (int64_t)members[t].size();
                if (sz <= edges[b] && (b == 0 || sz > edges[b - 1])) { ++cnt; r += sz; dsum += depth[t]; dmax = std::max(dmax, depth[t]); }
            }
            if (cnt) fprintf(stderr, "[ysolve]   rows<=%lld: %lld subtrees, %lld rows, sum depth %lld, max depth %d\n",
                             (long long)edges[b], (long long)cnt, (long long)r, (long long)dsum, dmax);
        }
    }
    // ---- top part: global levels, wide levels one launch each, narrow runs in one CTA
    int maxlev = -1;
    for (int32_t u : H.order) if (H.sub[u] < 0) maxlev = std::max(maxlev, (int)level[u]);
    S.levels = maxlev + 1;
    std::vector<std::vector<int32_t>> top_by_level(std::max(S.levels, 0));
    for (int32_t u : H.order) if (H.sub[u] < 0) top_by_level[level[u]].push_back(u);
    S.h_level_ptr.assign(S.levels + 1, (int64_t)slot_info.size());
    std::vector<int64_t> level_slots(std::max(S.levels, 1), 0);
    for (int l = 0; l < S.levels; ++l) {
        S.h_level_ptr[l] = (int64_t)slot_info.size();
        level_slots[l] = emit_level_slots(H, top_by_level[l], l, slot_rows, slot_info);
        S.h_level_ptr[l + 1] = (int64_t)slot_info.size();
    }
    S.n_slots = (int64_t)slot_info.size();
    int narrow_slots = kNarrowSlots;
    if (const char* e = getenv("CUADMM_SWEEP_NARROW_SLOTS")) narrow_slots = atoi(e);
    S.phases.clear();
    for (int l = 0; l < S.levels;) {
        if (level_slots[l] <= narrow_slots) {
            int e = l;
            while (e < S.levels && level_slots[e] <= narrow_slots) ++e;
            S.phases.push_back({true, l, e});
            l = e;
        } else {
            S.phases.push_back({false, l, l + 1});
            ++l;
        }
    }
    S.ptr.upload(H.ptr);
    std::vector<int32_t> dep(H.dep); if (dep.empty()) dep.push_back(0);
    std::vector<double> val(H.val); if (val.empty()) val.push_back(0.0);
    S.dep.upload(dep); S.val.upload(val);
    S.inv_diag.upload(H.inv_diag);
    if (slot_rows.empty()) { slot_rows.assign(8, -1); slot_info.push_back(0); }
    S.slot_rows.upload(slot_rows); S.slot_info.upload(slot_info);
    S.level_ptr.upload(S.h_level_ptr);
    if (sub_lvl_ptr.empty()) sub_lvl_ptr.push_back(0);
    S.sub_off.upload(sub_off); S.sub_lvl_ptr.upload(sub_lvl_ptr);
}

// Disjoint subtrees of the elimination tree (lead part only), each at most `cap` rows: v roots a
// subtree when its own subtree fits and its parent's does not (or the parent is in the dense tail).
static int64_t choose_subtrees(const CholFactor& F, int64_t n_lead, std::vector<int32_t>& sub) {
    const int64_t n = F.n;
    sub.assign(n, -1);
    int64_t cap = 12000;          // rows per subtree: its unknowns (+ up to 384 chain slots) live in shared memory next to the
                                  // 2 x 64 KB chunk ring: (12000 + 384) * 8 + 131136 bytes <= 227 KB
    if (const char* e = getenv("CUADMM_SWEEP_SUBTREE_CAP")) cap = atoll(e);
    if (cap <= 0) return 0;
    cap = std::min<int64_t>(cap, (int64_t)(232448 - kPkRing * kPkChunk - 64) / 8 - kPkChainMax);   // 227 KB of shared memory
    int64_t min_size = 2;         // (measured: peeling small subtrees off into extra top levels costs more than their CTAs)
    if (const char* e = getenv("CUADMM_SWEEP_SUBTREE_MIN")) min_size = atoll(e);
    std::vector<int64_t> size(n, 1);
    for (int64_t v = 0; v < n_lead; ++v) {
        const int32_t p = F.parent[v];
        if (p >= 0 && p < n_lead) size[p] += size[v];
    }
    int64_t n_sub = 0;
    for (int64_t v = n_lead - 1; v >= 0; --v) {
        const int32_t p = F.parent[v];
        const bool parent_top = (p < 0 || p >= n_lead || sub[p] < 0);
        if (!parent_top) { sub[v] = sub[p]; continue; }
        const bool parent_fits = (p >= 0 && p < n_lead && size[p] <= cap);
        if (size[v] <= cap && !parent_fits && size[v] >= min_size) sub[v] = (int32_t)n_sub++;
    }
    return n_sub;
}

// the 8-row blocks of rows [row0, row0 + nrows) (row0 a multiple of 8), counted from row0, longest rows first
static std::vector<int32_t> longest_first(const std::vector<double>& cost, int64_t row0, int64_t nrows) {
    std::vector<int32_t> b((size_t)std::max<int64_t>(1, (nrows + 7) / 8));
    std::iota(b.begin(), b.end(), 0);
    if (nrows > 0)
        std::stable_sort(b.begin(), b.end(), [&](int32_t x, int32_t y) { return cost[(row0 + 8 * x) >> 6] > cost[(row0 + 8 * y) >> 6]; });
    return b;
}

// Tile-run storage (TailMatrix) of L = P L22^-1 P^T (lower) or of L^T, from the occupancy flags of L.  Linv is L22^-1
// column-major in F's order, d_ipos P's map from new to old tail index.
static void pack_tail_matrix(int64_t r, const double* Linv, const int32_t* d_ipos, const std::vector<int>& flags, bool lower,
                             TailMatrix& T) {
    const int nt = (int)((r + 63) / 64);
    std::vector<int32_t> ptr(1, 0), col;
    std::vector<int64_t> off, tiles;       // tiles: (I, J, destination, row stride) for pack_tiles
    int64_t size = 0;
    T.cost.assign(nt, 0.0);
    for (int I = 0; I < nt; ++I) {
        const int J0 = lower ? 0 : I, J1 = lower ? I + 1 : nt;
        auto used = [&](int J) { return flags[lower ? (size_t)I * nt + J : (size_t)J * nt + I] != 0; };
        for (int J = J0; J < J1;) {
            if (!used(J)) { ++J; continue; }
            int E = J;
            while (E < J1 && used(E)) ++E;
            const int64_t w = (int64_t)(E - J) * 64;
            col.push_back(J * 64); col.push_back(E * 64);
            off.push_back(size);
            for (int K = J; K < E; ++K) { tiles.push_back(I); tiles.push_back(K); tiles.push_back(size + (K - J) * 64); tiles.push_back(w); }
            size += 64 * w;
            T.cost[I] += (double)w;
            J = E;
        }
        ptr.push_back((int32_t)(col.size() / 2));
    }
    if (col.empty()) { col.assign(2, 0); off.push_back(0); }
    T.val.alloc(std::max<int64_t>(size, 1));
    pack_tiles(r, Linv, d_ipos, !lower, tiles, T.val.p);
    T.tptr.upload(ptr); T.tcol.upload(col); T.toff.upload(off);
    T.order.upload(longest_first(T.cost, 0, r));
}

// Dense tail.  L22 is factored and inverted in F's order, so its pivots (and pivot floors) are those of that order; the
// finished inverse is then relabelled symmetrically, tail row i -> pos[i], and only its non-empty 64 x 64 tiles are
// stored.  L22^-1 (i, j) can be non-zero only when j is a descendant of i in the elimination tree: with pos a
// postorder of the tail's tree its few non-zeros gather in few tiles near the diagonal (C2b bench operator: 710 of
// 12,880 lower tiles instead of 8,054 in F's order), and the inverse stays lower triangular.  The numeric tile scan
// decides what is stored; if it finds a tile above the diagonal, pos falls back to the identity.
static void build_tail(cuadmm_ysolve_s& Y, const SymCsc& C, const CholFactor& F, std::vector<int32_t>& pos, int64_t* n_def) {
    const int64_t r = Y.n_tail;
    const int nt = (int)((r + 63) / 64);
    DevBuf<double> Linv;                   // r x r: init-time scratch, freed on return
    build_dense_tail(C, F, Y.n_lead, r, Linv, n_def);
    DevBuf<int32_t> d_ipos;
    std::vector<int> flags;
    auto scan = [&]() {
        std::vector<int32_t> ipos(r);
        for (int64_t i = 0; i < r; ++i) ipos[pos[i]] = (int32_t)i;
        d_ipos.upload(ipos);
        tile_occupancy(r, Linv.p, d_ipos.p, flags);
    };
    auto lower_used = [&]() {
        int64_t used = 0;
        for (int I = 0; I < nt; ++I) for (int J = 0; J <= I; ++J) used += flags[(size_t)I * nt + J];
        return used;
    };
    const bool verbose = getenv("CUADMM_YSOLVE_VERBOSE") != nullptr;
    int64_t used_before = -1;
    if (verbose) {
        const std::vector<int32_t> keep(pos);
        std::iota(pos.begin(), pos.end(), 0);
        scan();
        used_before = lower_used();
        pos = keep;
    }
    scan();
    bool upper = false;
    for (int I = 0; I < nt && !upper; ++I) for (int J = I + 1; J < nt; ++J) if (flags[(size_t)I * nt + J]) { upper = true; break; }
    if (upper) {
        std::iota(pos.begin(), pos.end(), 0);
        scan();
    }
    if (verbose) {
        const int64_t lower = (int64_t)nt * (nt + 1) / 2, used = lower_used();
        fprintf(stderr, "[ysolve] dense tail %lld: non-zero lower 64x64 tiles of L22^-1: %lld of %lld (%.1f%%) in the tail order, "
                "%lld (%.1f%%) stored%s\n", (long long)r, (long long)used_before, (long long)lower,
                100.0 * (double)used_before / (double)lower, (long long)used, 100.0 * (double)used / (double)lower,
                upper ? " (postorder left a tile above the diagonal: tail order kept)" : "");
    }
    pack_tail_matrix(r, Linv.p, d_ipos.p, flags, true, Y.tail[0]);
    pack_tail_matrix(r, Linv.p, d_ipos.p, flags, false, Y.tail[1]);
}

cuadmm_ysolve_s* ysolve_create(int64_t m, int64_t vec_len, int64_t nnz, const int32_t* rowptr, const int32_t* colind,
                               const double* val, double eps, int device) {
    CUADMM_REQUIRE(m >= 0 && vec_len >= 0 && nnz >= 0, "negative dimension");
    CUADMM_REQUIRE(rowptr && (nnz == 0 || (colind && val)), "null argument");
    CUADMM_REQUIRE(rowptr[0] == 0 && rowptr[m] == nnz, "rowptr does not span nnz");
    int cnt = 0;
    if (cudaGetDeviceCount(&cnt) != cudaSuccess || cnt == 0) {
        cudaGetLastError();
        throw Error(CUADMM_ENODEVICE, "no CUDA device available; the y-solve has no CPU fallback");
    }
    CUADMM_REQUIRE(device >= 0 && device < cnt, "device index out of range");
    std::unique_ptr<cuadmm_ysolve_s> Y(new cuadmm_ysolve_s());
    Y->device = device; Y->m = m;
    DeviceGuard g(device);

    // ---- host analysis (CUADMM_YSOLVE_VERBOSE prints the wall time of every phase)
    const bool vtime = getenv("CUADMM_YSOLVE_VERBOSE") != nullptr;
    auto tp0 = std::chrono::steady_clock::now();
    auto lap = [&](const char* what) {
        if (!vtime) return;
        const auto t = std::chrono::steady_clock::now();
        fprintf(stderr, "[ysolve] init %-28s %8.1f ms\n", what, std::chrono::duration<double, std::milli>(t - tp0).count());
        tp0 = t;
    };
    SymCsc M = form_aat(m, vec_len, rowptr, colind, val, eps);
    lap("A A^T");
    Y->nnz_aat = M.p[m];
    CholFactor F;
    SymCsc C;
    const int64_t n_lead = order_tail_last(M, F, C);
    const int64_t n_tail = m - n_lead;
    lap("ordering + symbolic (tail last)");
    chol_numeric(C, F, n_lead);
    lap("numeric (sparse lead part)");
    Y->n_lead = n_lead; Y->n_tail = n_tail;
    Y->nnz_L = F.nnz();
    Y->n_deficient = F.n_deficient;

    // ---- dense tail: S = M22 - L21 L21^T, Cholesky, explicit inverse (all on the device), stored relabelled
    std::vector<int32_t> pos(n_tail);
    std::iota(pos.begin(), pos.end(), 0);
    if (n_tail > 0) {
        const char* e = getenv("CUADMM_YSOLVE_TAIL_POSTORDER");     // "0": keep the tail order (probe of the relabelling)
        if (!(e && atoi(e) == 0)) pos = tail_postorder(F, n_lead);
        int64_t tail_def = 0;
        build_tail(*Y, C, F, pos, &tail_def);
        Y->n_deficient += tail_def;
        Y->tail_tmp.alloc(n_tail);
        lap("dense tail (GPU)");
    }
    // The sweeps and perm use the relabelled tail: unknown n_lead + i of F is n_lead + pos[i] here.  Lead unknowns keep
    // their ids, every row keeps its entries in the same order, so the sweeps do the arithmetic of F's order.
    auto relabel = [&](int32_t u) { return u < n_lead ? u : (int32_t)(n_lead + pos[u - n_lead]); };
    Y->h_perm.resize(m);
    for (int64_t k = 0; k < m; ++k) Y->h_perm[relabel((int32_t)k)] = F.perm[k];
    Y->perm.upload(Y->h_perm);

    std::vector<int32_t> sub;
    const int64_t n_sub = choose_subtrees(F, n_lead, sub);
    // ---- forward sweep: rows of L (lead rows solve, tail rows accumulate t2 = b2 - L21 z1)
    {
        HostSweep H;
        H.n = m;
        H.ptr.assign(m + 1, 0);
        for (int64_t j = 0; j < n_lead; ++j)
            for (int64_t p = F.Lp[j] + 1; p < F.Lp[j + 1]; ++p) H.ptr[relabel(F.Li[p]) + 1]++;
        for (int64_t i = 0; i < m; ++i) H.ptr[i + 1] += H.ptr[i];
        H.dep.resize(H.ptr[m]); H.val.resize(H.ptr[m]);
        std::vector<int64_t> nx(H.ptr.begin(), H.ptr.end() - 1);
        for (int64_t j = 0; j < n_lead; ++j)
            for (int64_t p = F.Lp[j] + 1; p < F.Lp[j + 1]; ++p) {
                const int64_t q = nx[relabel(F.Li[p])]++;
                H.dep[q] = (int32_t)j; H.val[q] = F.Lx[p];
            }
        H.inv_diag.assign(m, 1.0);
        for (int64_t i = 0; i < n_lead; ++i) H.inv_diag[i] = 1.0 / F.Lx[F.Lp[i]];
        H.order.resize(m);
        std::iota(H.order.begin(), H.order.end(), 0);
        H.sub = sub; H.n_sub = n_sub; H.subtrees_first = true;
        H.gather = &Y->h_perm;
        upload_sweep(H, Y->fwd);
    }
    // ---- backward sweep: columns of L as rows of L^T, lead unknowns only
    {
        HostSweep H;
        H.n = m;
        H.ptr.assign(m + 1, 0);
        for (int64_t j = 0; j < n_lead; ++j) H.ptr[j + 1] = F.Lp[j + 1] - F.Lp[j] - 1;
        for (int64_t i = 0; i < m; ++i) H.ptr[i + 1] += H.ptr[i];
        H.dep.resize(H.ptr[m]); H.val.resize(H.ptr[m]);
        for (int64_t j = 0; j < n_lead; ++j) {
            int64_t q = H.ptr[j];
            for (int64_t p = F.Lp[j] + 1; p < F.Lp[j + 1]; ++p, ++q) { H.dep[q] = relabel(F.Li[p]); H.val[q] = F.Lx[p]; }
        }
        H.inv_diag.assign(m, 1.0);
        for (int64_t i = 0; i < n_lead; ++i) H.inv_diag[i] = 1.0 / F.Lx[F.Lp[i]];
        H.order.resize(n_lead);
        for (int64_t j = 0; j < n_lead; ++j) H.order[j] = (int32_t)(n_lead - 1 - j);
        // tail unknowns are final before the backward sweep starts: give them their own "part"
        H.sub = sub;
        for (int64_t i = n_lead; i < m; ++i) H.sub[i] = -2;
        H.n_sub = n_sub; H.subtrees_first = false;
        H.out_perm = &Y->h_perm;
        upload_sweep(H, Y->bwd);
    }
    lap("pack + upload sweeps");
    Y->z.alloc(std::max<int64_t>(m, 1));
    Y->x.alloc(std::max<int64_t>(m, 1));

    Y->launches_per_solve = (int)(Y->fwd.phases.size() + Y->bwd.phases.size()) + (n_tail > 0 ? 2 : 0) +
                            (Y->fwd.n_sub_cta > 0 ? 2 : 0) + (Y->fwd.n_sub_warp > 0 ? 2 : 0) + (Y->fwd.n_sub_pack > 0 ? 2 : 0) +
                            (Y->fwd.pk_rows > 0 ? 2 : 0);
    CUADMM_CUDA(cudaStreamCreateWithFlags(&Y->streams.side, cudaStreamNonBlocking));
    CUADMM_CUDA(cudaEventCreateWithFlags(&Y->streams.fork, cudaEventDisableTiming));
    CUADMM_CUDA(cudaEventCreateWithFlags(&Y->streams.join, cudaEventDisableTiming));
    Y->alg_bytes = 2 * (12 * Y->nnz_L + 8 * m) + 24 * m;
    CUADMM_CUDA(cudaDeviceSynchronize());
    return Y.release();
}

}  // namespace cuadmm

using namespace cuadmm;

cuadmm_ysolve_s::~cuadmm_ysolve_s() {
    if (streams.fork) cudaEventDestroy(streams.fork);
    if (streams.join) cudaEventDestroy(streams.join);
    if (streams.side) cudaStreamDestroy(streams.side);
}

void cuadmm_ysolve_s::enable_peer(const PeerComm* pc, size_t off_tmp, size_t off_x) {
    peer = pc;
    peer_tmp = pc->ptrs(off_tmp);
    peer_x = pc->ptrs(off_x);
    tail_tmp_p = pc->local<double>(off_tmp);
    x_p = pc->local<double>(off_x);
    if (n_tail > 0 && pc->world > 1) launches_per_solve += 1;     // tail_scatter_kernel
    split_tail_rows(pc->world, pc->rank);
}

// rows of each tail GEMV split into `world` contiguous ranges of equal work (columns read)
void cuadmm_ysolve_s::split_tail_rows(int world, int rank) {
    for (int k = 0; k < 2; ++k) {
        const std::vector<double>& c = tail[k].cost;
        double total = 0.0;
        for (int64_t i = 0; i < n_tail; ++i) total += c[i >> 6] + 32.0;
        std::vector<int64_t> cut(world + 1, n_tail);
        cut[0] = 0;
        double acc = 0.0;
        int q = 1;
        for (int64_t i = 0; i < n_tail && q < world; ++i) {
            acc += c[i >> 6] + 32.0;
            while (q < world && acc >= total * q / world) cut[q++] = std::min<int64_t>(n_tail, (i + 1 + 7) / 8 * 8);   // CTA = 8 rows
        }
        tail_row0[k] = cut[rank]; tail_row1[k] = cut[rank + 1];
        tail[k].rank_order.upload(longest_first(c, tail_row0[k], tail_row1[k] - tail_row0[k]));
    }
    // scratch of the split-column GEMV (allocated here: solve() may run inside a stream capture)
    const int64_t nrb = std::max<int64_t>(1, (std::max(tail_row1[0] - tail_row0[0], tail_row1[1] - tail_row0[1]) + 7) / 8);
    split_part.alloc(nrb * 8 * 8);
    split_count.alloc(nrb);
    split_count.zero();
    CUADMM_CUDA(cudaDeviceSynchronize());
}

void cuadmm_ysolve_s::solve(const double* d_rhs_, double* d_y_, cudaStream_t st) {
    if (m == 0) return;
    double* xv = x_p ? x_p : x.p;
    double* tmpv = tail_tmp_p ? tail_tmp_p : tail_tmp.p;
    // forward: z = L11^-1 P rhs (lead), z_tail = P rhs - L21 z_lead
    launch_sweep(fwd, d_rhs_, perm.p, z.p, nullptr, nullptr, done_flag, st, streams);
    auto mark = [&](int tag) {
        if (!prof_ev) return;
        cudaEvent_t ev;
        CUADMM_CUDA(cudaEventCreate(&ev));
        CUADMM_CUDA(cudaEventRecord(ev, st));
        prof_ev->push_back(ev); prof_tag->push_back(tag);
    };
    // split-column GEMV over this rank's rows: enough CTAs per row block to fill the GPU twice
    auto gemv_split = [&](const TailMatrix& T, const double* in, double* out, int64_t r0, int64_t nrows_, int npush,
                          const PeerView& pv, const PeerPtrs& outp) {
        const int64_t nrb = std::max<int64_t>(1, (nrows_ + 7) / 8);
        int splits = (int)std::min<int64_t>(8, std::max<int64_t>(1, (2 * 148 + nrb - 1) / nrb));
        CUADMM_REQUIRE(split_part.n >= nrb * 8 * 8 && split_count.n >= nrb && T.rank_order.n >= nrb,
                       "internal: split-column GEMV scratch too small");
        tail_gemv_kernel<<<(unsigned)(nrb * splits), 256, 0, st>>>(n_tail, T.val.p, in, out, T.tptr.p, T.tcol.p, T.toff.p,
            T.rank_order.p, nullptr, nullptr, 0, done_flag, r0, nrows_, npush, pv, outp, PeerPtrs(), splits, split_part.p,
            split_count.p);
    };
    if (n_tail > 0) {
        mark(20);
        // x_tail = L22^-T L22^-1 z_tail, scattered into y
        if (!peer || peer->world == 1) {
            const int blocks = (int)((n_tail + 7) / 8);
            // whole matrix on one GPU: row per warp streams at 69 % of the HBM peak (ncu), the split-column kernel at 55 %
            tail_gemv_row_kernel<<<blocks, 256, 0, st>>>(n_tail, tail[0].val.p, z.p + n_lead, tmpv, tail[0].tptr.p, tail[0].tcol.p,
                                                         tail[0].toff.p, tail[0].order.p, nullptr, nullptr, 0, done_flag);
            tail_gemv_row_kernel<<<blocks, 256, 0, st>>>(n_tail, tail[1].val.p, tmpv, xv + n_lead, tail[1].tptr.p, tail[1].tcol.p,
                                                         tail[1].toff.p, tail[1].order.p, d_y_, perm.p, n_lead, done_flag);
        } else {
            PeerPtrs pxt = peer_x;
            for (int q = 0; q < peer->world; ++q) pxt.p[q] += n_lead;
            const PeerView pv = peer->view();
            const int64_t n0 = tail_row1[0] - tail_row0[0], n1 = tail_row1[1] - tail_row0[1];
            gemv_split(tail[0], z.p + n_lead, tmpv, tail_row0[0], n0, peer->world, pv, peer_tmp);
            gemv_split(tail[1], tmpv, xv + n_lead, tail_row0[1], n1, peer->world, pv, pxt);
            tail_scatter_kernel<<<(int)((n_tail + 255) / 256), 256, 0, st>>>(n_tail, xv + n_lead, perm.p, n_lead, d_y_, done_flag);
        }
        CUADMM_CUDA(cudaGetLastError());
        mark(21);
    }
    // backward: x_lead = L11^-T (z_lead - L21^T x_tail), scattered into y
    launch_sweep(bwd, z.p, nullptr, xv, d_y_, perm.p, done_flag, st, streams);
}

extern "C" {

int cuadmm_ysolve_create(int64_t m, int64_t vec_len, int64_t nnz, const int32_t* h_A_rowptr, const int32_t* h_A_colind,
                         const double* h_A_val, double eps, int device, cuadmm_ysolve_t** out) {
    return guarded([&] {
        CUADMM_REQUIRE(out != nullptr, "out is null");
        *out = nullptr;
        *out = ysolve_create(m, vec_len, nnz, h_A_rowptr, h_A_colind, h_A_val, eps, device);
    });
}

void cuadmm_ysolve_destroy(cuadmm_ysolve_t* ys) { delete ys; }

int cuadmm_ysolve(cuadmm_ysolve_t* ys, const double* d_rhs, double* d_y, void* stream) {
    return guarded([&] {
        CUADMM_REQUIRE(ys && d_rhs && d_y, "null argument");
        DeviceGuard g(ys->device);
        ys->solve(d_rhs, d_y, (cudaStream_t)stream);
    });
}

// debug: timeline[4*t..] = globaltimer stamps (start, after prologue, after levels, end) of CTA t of the
// packed kernel of the last solve (which: 0 forward, 1 backward); meta[3*t..] = chunks, rows, depth.
// Needs CUADMM_YSOLVE_TIMELINE=1 at create time.  Returns the CTA count through *n.
int cuadmm_debug_ysolve_timeline(cuadmm_ysolve_t* ys, int which, long long* timeline, long long* meta, int64_t cap, int64_t* n) {
    return guarded([&] {
        CUADMM_REQUIRE(ys && n, "null argument");
        DeviceGuard g(ys->device);
        const cuadmm::TriSweep& S = which ? ys->bwd : ys->fwd;
        *n = S.pk_timeline.n / 4;
        if (!timeline || cap < *n || *n == 0) return;
        CUADMM_CUDA(cudaDeviceSynchronize());
        CUADMM_CUDA(cudaMemcpy(timeline, S.pk_timeline.p, sizeof(long long) * 4 * (size_t)*n, cudaMemcpyDeviceToHost));
        if (meta) std::copy(S.pk_timeline_meta.begin(), S.pk_timeline_meta.end(), meta);
    });
}

int cuadmm_ysolve_host(cuadmm_ysolve_t* ys, const double* h_rhs, double* h_y) {
    return guarded([&] {
        CUADMM_REQUIRE(ys && h_rhs && h_y, "null argument");
        DeviceGuard g(ys->device);
        if (ys->d_rhs.n != ys->m) { ys->d_rhs.alloc(std::max<int64_t>(ys->m, 1)); ys->d_y.alloc(std::max<int64_t>(ys->m, 1)); }
        ys->d_rhs.upload(h_rhs, ys->m);
        ys->solve(ys->d_rhs.p, ys->d_y.p, 0);
        ys->d_y.download(h_y, ys->m);
        CUADMM_CUDA(cudaStreamSynchronize(0));
    });
}

int cuadmm_ysolve_stats(const cuadmm_ysolve_t* ys, int64_t out[8]) {
    return guarded([&] {
        CUADMM_REQUIRE(ys && out, "null argument");
        out[0] = ys->nnz_aat; out[1] = ys->nnz_L; out[2] = std::max(ys->fwd.levels, ys->bwd.levels);
        out[3] = ys->n_tail; out[4] = ys->launches_per_solve; out[5] = ys->alg_bytes;
        out[6] = ys->n_deficient; out[7] = ys->fwd.n_sub * 100000 + ys->fwd.sub_depth;
    });
}

int cuadmm_ysolve_perm(const cuadmm_ysolve_t* ys, int32_t* perm) {
    return guarded([&] {
        CUADMM_REQUIRE(ys && perm, "null argument");
        std::copy(ys->h_perm.begin(), ys->h_perm.end(), perm);
    });
}

}  // extern "C"
