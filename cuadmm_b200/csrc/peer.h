// peer.h — peer-memory transport of the sharded solver: every rank (one process per GPU) owns one
// device arena, exports it with CUDA IPC and maps the arenas of all other ranks, so kernels exchange data
// with plain loads/stores over NVLink / NVSwitch and synchronise through system-scope flags — the
// collective is part of the kernel that produces or consumes the data (SpMV rows are stored straight
// into the staging area of the rank that reduces them, reduced slices and dense-tail GEMV rows are
// stored straight into every peer's copy).  Replaces the hub-and-spoke cudaMemcpyPeerAsync of
// src/duo_solver.cu:517-565 and the NCCL all-reduce calls of round 1.
//
// Handshake protocol (device side, see peer_enter / peer_leave): a kernel that pushes data to its peers
//   1. [enter]  tells every peer "I reached handshake e" and waits until every peer said the same: all
//               earlier pushes addressed to this rank have landed and every peer is done reading what
//               this kernel is about to overwrite;
//   2. pushes (stores into peer arenas);
//   3. [leave]  the last CTA tells every peer "my pushes of handshake e are complete" and waits for the
//               same message from every peer: when the kernel retires, this rank's copies are complete.
// e is a device-resident counter that every rank advances identically (all ranks run the same launch
// sequence), so the protocol is CUDA-graph friendly: nothing in the kernel arguments changes per launch.
// Spin loops give up after a time-out and raise an error word the host checks (no hung GPU).
#pragma once
#include "common.h"

namespace cuadmm {

constexpr int kMaxPeers = 8;

struct PeerView {
    int rank = 0, world = 1;
    unsigned long long* epoch = nullptr;       // private: handshakes completed
    unsigned int* cta_count = nullptr;         // private: CTAs of the running kernel that finished pushing
    int* err = nullptr;                        // private: 1 after a time-out
    unsigned long long timeout_ns = 0;
    unsigned long long* ready[kMaxPeers] = {}; // ready[q] + r : flag in rank q's arena written by rank r
    unsigned long long* fin[kMaxPeers] = {};
};

// the same buffer in every rank's arena
struct PeerPtrs {
    double* p[kMaxPeers] = {};
};

struct PeerComm {
    int rank = 0, world = 1, device = 0;
    char* base[kMaxPeers] = {};
    size_t bytes = 0, used = 0;
    DevBuf<unsigned long long> d_epoch;
    DevBuf<unsigned int> d_count;
    DevBuf<int> d_err;
    size_t off_ready = 0, off_fin = 0, off_scal_rd = 0, off_scal_rp = 0, off_scal_chk = 0;
    unsigned long long timeout_ns = 120ull * 1000000000ull;   // ranks may reach their first handshake seconds apart (init skew)

    ~PeerComm();
    // collective: every rank calls it with the same id and arena size
    void init(int rank, int world, const char id[128], int device, size_t arena_bytes);
    // bump allocation inside the arena; every rank must issue the same sequence of calls
    size_t alloc(size_t nbytes);
    template <class T> T* at(int q, size_t off) const { return reinterpret_cast<T*>(base[q] + off); }
    template <class T> T* local(size_t off) const { return at<T>(rank, off); }
    PeerPtrs ptrs(size_t off) const { PeerPtrs r; for (int q = 0; q < world; ++q) r.p[q] = at<double>(q, off); return r; }
    PeerView view() const;
    // throws if a device-side handshake timed out (call after a stream synchronisation)
    void check(cudaStream_t stream);
    static size_t control_bytes();
};

void make_unique_id(char out[128]);

#ifdef __CUDACC__
__device__ __forceinline__ void peer_st_release(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long peer_ld_acquire(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long peer_now_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ void peer_spin(const PeerView& pv, const unsigned long long* flag, unsigned long long e) {
    if (peer_ld_acquire(flag) >= e) return;
    const unsigned long long t0 = peer_now_ns();
    while (peer_ld_acquire(flag) < e) {
        __nanosleep(64);
        if (peer_now_ns() - t0 > pv.timeout_ns) { *pv.err = 1; break; }
    }
}
// handshake number of the running kernel (same value in every CTA: the counter only moves in peer_leave,
// after every CTA has passed it)
__device__ __forceinline__ unsigned long long peer_epoch(const PeerView& pv) {
    return *reinterpret_cast<volatile unsigned long long*>(pv.epoch) + 1ull;
}
// all threads of all CTAs
__device__ __forceinline__ void peer_enter(const PeerView& pv, unsigned long long e) {
    if (blockIdx.x == 0 && (int)threadIdx.x < pv.world) {
        __threadfence_system();
        peer_st_release(pv.ready[threadIdx.x] + pv.rank, e);
    }
    if ((int)threadIdx.x < pv.world) peer_spin(pv, pv.ready[pv.rank] + threadIdx.x, e);
    __syncthreads();
}
// all threads of all CTAs, after their last push
__device__ __forceinline__ void peer_leave(const PeerView& pv, unsigned long long e) {
    __shared__ int s_last;
    // the CTA's remote stores are ordered before thread 0's fence by the barrier (cumulativity): one fence per CTA, and
    // only at device scope — the system-scope release comes once, from the last CTA, after it has observed all the others
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        s_last = (atomicAdd(pv.cta_count, 1u) == gridDim.x - 1u) ? 1 : 0;
    }
    __syncthreads();
    if (!s_last) return;
    if ((int)threadIdx.x < pv.world) {
        __threadfence_system();
        peer_st_release(pv.fin[threadIdx.x] + pv.rank, e);
        peer_spin(pv, pv.fin[pv.rank] + threadIdx.x, e);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        *pv.cta_count = 0u;
        *reinterpret_cast<volatile unsigned long long*>(pv.epoch) = e;
        __threadfence();
    }
}
#endif

}  // namespace cuadmm
