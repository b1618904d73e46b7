// peer.cu — see peer.h: CUDA-IPC arena exchange through a POSIX shared-memory board + the slice
// reduction kernel of the sharded solver.
#include "peer.h"
#include "peer_kernels.h"
#include <fcntl.h>
#include <string.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
#include <atomic>
#include <chrono>
#include <thread>

namespace cuadmm {

namespace {
struct Board {
    std::atomic<int> posted[kMaxPeers];
    std::atomic<int> opened[kMaxPeers];
    cudaIpcMemHandle_t handle[kMaxPeers];
    unsigned long long bytes[kMaxPeers];
};

std::string board_name(const char id[128]) {
    unsigned long long h = 1469598103934665603ull;   // FNV-1a over the job id
    for (int i = 0; i < 128; ++i) { h ^= (unsigned char)id[i]; h *= 1099511628211ull; }
    char buf[64];
    snprintf(buf, sizeof buf, "/cuadmm_b200_%016llx", h);
    return buf;
}

template <class F>
void wait_for(F&& cond, const char* what) {
    const auto t0 = std::chrono::steady_clock::now();
    while (!cond()) {
        std::this_thread::sleep_for(std::chrono::microseconds(200));
        if (std::chrono::steady_clock::now() - t0 > std::chrono::seconds(180))
            throw Error(CUADMM_ENCCL, std::string("peer rendezvous timed out waiting for ") + what);
    }
}
}  // namespace

void make_unique_id(char out[128]) {
    int fd = open("/dev/urandom", O_RDONLY);
    bool ok = false;
    if (fd >= 0) { ok = read(fd, out, 128) == 128; close(fd); }
    if (!ok) {
        unsigned long long s = (unsigned long long)std::chrono::steady_clock::now().time_since_epoch().count() ^ ((unsigned long long)getpid() << 32);
        for (int i = 0; i < 128; ++i) { s = s * 6364136223846793005ull + 1442695040888963407ull; out[i] = (char)(s >> 56); }
    }
}

size_t PeerComm::control_bytes() { return 4096; }

void PeerComm::init(int rank_, int world_, const char id[128], int device_, size_t arena_bytes) {
    CUADMM_REQUIRE(world_ >= 1 && world_ <= kMaxPeers, "peer transport supports up to 8 ranks (one NVSwitch box)");
    rank = rank_; world = world_; device = device_;
    CUADMM_CUDA(cudaSetDevice(device));
    bytes = (arena_bytes + control_bytes() + 4095) / 4096 * 4096;
    void* mine = nullptr;
    CUADMM_CUDA(cudaMalloc(&mine, bytes));
    CUADMM_CUDA(cudaMemset(mine, 0, bytes));
    CUADMM_CUDA(cudaDeviceSynchronize());
    base[rank] = static_cast<char*>(mine);
    d_epoch.alloc(1); d_count.alloc(2); d_err.alloc(1);
    d_epoch.zero(); d_count.zero(); d_err.zero();
    if (const char* e = getenv("CUADMM_PEER_TIMEOUT_S")) { const double s = atof(e); if (s > 0) timeout_ns = (unsigned long long)(s * 1e9); }
    // control block: ready / fin flags (one 8-byte word per writer rank) and the two scalar boards (2 doubles per rank)
    off_ready = 0; off_fin = 1024; off_scal_rd = 2048; off_scal_rp = 2048 + 512;
    used = control_bytes();
    if (world > 1) {
        const std::string name = board_name(id);
        int fd = shm_open(name.c_str(), O_CREAT | O_RDWR, 0600);
        if (fd < 0) throw Error(CUADMM_ENCCL, "shm_open failed for the peer rendezvous board " + name);
        if (ftruncate(fd, sizeof(Board)) != 0) { close(fd); throw Error(CUADMM_ENCCL, "ftruncate failed for the peer rendezvous board"); }
        Board* b = static_cast<Board*>(mmap(nullptr, sizeof(Board), PROT_READ | PROT_WRITE, MAP_SHARED, fd, 0));
        close(fd);
        if (b == MAP_FAILED) throw Error(CUADMM_ENCCL, "mmap failed for the peer rendezvous board");
        try {
            CUADMM_CUDA(cudaIpcGetMemHandle(&b->handle[rank], mine));
            b->bytes[rank] = bytes;
            b->posted[rank].store(1, std::memory_order_release);
            for (int q = 0; q < world; ++q) {
                if (q == rank) continue;
                wait_for([&] { return b->posted[q].load(std::memory_order_acquire) == 1; }, "a peer's IPC handle");
                if (b->bytes[q] != bytes) throw Error(CUADMM_EINVAL, "ranks disagree on the peer arena size (different problems per rank?)");
                void* p = nullptr;
                CUADMM_CUDA(cudaIpcOpenMemHandle(&p, b->handle[q], cudaIpcMemLazyEnablePeerAccess));
                base[q] = static_cast<char*>(p);
            }
            b->opened[rank].store(1, std::memory_order_release);
            for (int q = 0; q < world; ++q)
                wait_for([&] { return b->opened[q].load(std::memory_order_acquire) == 1; }, "the peers to map this rank's arena");
        } catch (...) {
            munmap(b, sizeof(Board));
            shm_unlink(name.c_str());
            throw;
        }
        munmap(b, sizeof(Board));
        if (rank == 0) shm_unlink(name.c_str());
    }
}

PeerComm::~PeerComm() {
    cudaSetDevice(device);
    for (int q = 0; q < world; ++q) {
        if (!base[q]) continue;
        if (q == rank) cudaFree(base[q]); else cudaIpcCloseMemHandle(base[q]);
    }
}

size_t PeerComm::alloc(size_t nbytes) {
    const size_t off = (used + 255) / 256 * 256;
    if (off + nbytes > bytes) throw Error(CUADMM_ENOMEM, "peer arena exhausted");
    used = off + nbytes;
    return off;
}

PeerView PeerComm::view() const {
    PeerView v;
    v.rank = rank; v.world = world;
    v.epoch = d_epoch.p; v.cta_count = d_count.p; v.err = d_err.p;
    v.timeout_ns = timeout_ns;
    for (int q = 0; q < world; ++q) {
        v.ready[q] = at<unsigned long long>(q, off_ready);
        v.fin[q] = at<unsigned long long>(q, off_fin);
    }
    return v;
}

void PeerComm::check(cudaStream_t stream) {
    int e = 0;
    CUADMM_CUDA(cudaMemcpyAsync(&e, d_err.p, sizeof(int), cudaMemcpyDeviceToHost, stream));
    CUADMM_CUDA(cudaStreamSynchronize(stream));
    if (e) throw Error(CUADMM_ENCCL, "peer handshake timed out on the device (a rank died or diverged)");
}

// ------------------------------------------------------------------------------------------
// kernels
// ------------------------------------------------------------------------------------------
static constexpr int kRedThreads = 256;

// Slice reduction fused with its consumer.  The producers (SpMV rows, spmv.cu mode 5) have already stored
// partial row r_g[i] of rank g into stage[owner(i)][g][i - owner(i)*slice].  This rank sums its slice over
// g in rank order (every rank gets bit-identical sums), applies the consumer and stores the result slice into
// EVERY rank's copy of the output vector:
//   mode 0: out = sum                              (asmc = -A (S - C))
//   mode 1: out = b - sum (Rp); per-slice sums of |normA .* Rp|^2 and <b, y> go with the two local scalars of
//           K7 (sum_rd pairs) to every rank's scalar boards (scalar_update_kernel adds them in rank order)
__global__ void __launch_bounds__(kRedThreads) peer_reduce_kernel(PeerView pv, int mode, int64_t count, int64_t slice,
        const double* stage, PeerPtrs out, const double* __restrict__ b, const double* __restrict__ normA,
        const double* __restrict__ y, const double* __restrict__ part_rd, int n_rd, double* cta_part,
        PeerPtrs scal_rd, PeerPtrs scal_rp, const int* __restrict__ done_flag) {
    if (done_flag && *done_flag) return;
    const unsigned long long e = peer_epoch(pv);
    peer_enter(pv, e);
    const int64_t j0 = (int64_t)pv.rank * slice;
    const int64_t len = max((int64_t)0, min(slice, count - j0));
    double a0 = 0.0, a1 = 0.0;
    for (int64_t j = (int64_t)blockIdx.x * kRedThreads + threadIdx.x; j < len; j += (int64_t)gridDim.x * kRedThreads) {
        double s = 0.0;
        for (int g = 0; g < pv.world; ++g) s += __ldcg(stage + (int64_t)g * slice + j);   // written by the peers: L2 is the point of coherence
        const int64_t i = j0 + j;
        double v = s;
        if (mode == 1) {
            const double bi = b[i];
            v = bi - s;
            const double t = normA[i] * v;
            a0 = fma(t, t, a0);
            a1 = fma(bi, y[i], a1);
        }
        for (int q = 0; q < pv.world; ++q) out.p[q][i] = v;
    }
    if (mode == 1) {
        __shared__ double red[2][kRedThreads / 32];
        __shared__ int s_islast;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { a0 += __shfl_xor_sync(0xffffffffu, a0, o); a1 += __shfl_xor_sync(0xffffffffu, a1, o); }
        if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = a0; red[1][threadIdx.x >> 5] = a1; }
        __syncthreads();
        if (threadIdx.x == 0) {
            double s0 = 0.0, s1 = 0.0;
            for (int k = 0; k < kRedThreads / 32; ++k) { s0 += red[0][k]; s1 += red[1][k]; }
            cta_part[2 * blockIdx.x] = s0; cta_part[2 * blockIdx.x + 1] = s1;
            __threadfence();
            // the CTA that finds every other partial written folds them in a fixed order and publishes the scalars
            s_islast = (atomicAdd(pv.cta_count + 1, 1u) == gridDim.x - 1u) ? 1 : 0;
        }
        __syncthreads();
        if (s_islast && threadIdx.x == 0) {
            __threadfence();
            double s0 = 0.0, s1 = 0.0, r0 = 0.0, r1 = 0.0;
            for (unsigned k = 0; k < gridDim.x; ++k) { s0 += __ldcg(cta_part + 2 * k); s1 += __ldcg(cta_part + 2 * k + 1); }
            for (int k = 0; k < n_rd; ++k) { r0 += part_rd[2 * k]; r1 += part_rd[2 * k + 1]; }
            for (int q = 0; q < pv.world; ++q) {
                scal_rd.p[q][2 * pv.rank] = r0; scal_rd.p[q][2 * pv.rank + 1] = r1;
                scal_rp.p[q][2 * pv.rank] = s0; scal_rp.p[q][2 * pv.rank + 1] = s1;
            }
            pv.cta_count[1] = 0u;
        }
    }
    peer_leave(pv, e);
}

// gather by owner: every rank stores its owned svec ranges into every rank's full-length vector
__global__ void __launch_bounds__(kRedThreads) peer_scatter_full_kernel(PeerView pv, int64_t nloc, const double* __restrict__ local,
        const int64_t* __restrict__ loc2glob, PeerPtrs full) {
    const unsigned long long e = peer_epoch(pv);
    peer_enter(pv, e);
    for (int64_t i = (int64_t)blockIdx.x * kRedThreads + threadIdx.x; i < nloc; i += (int64_t)gridDim.x * kRedThreads) {
        const double v = local[i];
        const int64_t g = loc2glob[i];
        for (int q = 0; q < pv.world; ++q) full.p[q][g] = v;
    }
    peer_leave(pv, e);
}

static int red_grid(int64_t n, int device) {
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    return (int)std::max<int64_t>(1, std::min<int64_t>((n + kRedThreads * 2 - 1) / (kRedThreads * 2), (int64_t)sms));
}

int peer_reduce_grid(const PeerComm& pc, int64_t slice) { return red_grid(slice, pc.device); }

void peer_reduce_launch(const PeerComm& pc, int mode, int64_t count, int64_t slice, const double* stage, const PeerPtrs& out,
                        const double* b, const double* normA, const double* y, const double* part_rd, int n_rd, double* cta_part,
                        const int* done_flag, cudaStream_t stream) {
    const int grid = red_grid(slice, pc.device);
    peer_reduce_kernel<<<grid, kRedThreads, 0, stream>>>(pc.view(), mode, count, slice, stage, out, b, normA, y, part_rd, n_rd,
                                                         cta_part, pc.ptrs(pc.off_scal_rd), pc.ptrs(pc.off_scal_rp), done_flag);
    CUADMM_CUDA(cudaGetLastError());
}

void peer_scatter_full_launch(const PeerComm& pc, int64_t nloc, const double* local, const int64_t* loc2glob, const PeerPtrs& full,
                              cudaStream_t stream) {
    const int grid = red_grid(std::max<int64_t>(nloc, 1), pc.device);
    peer_scatter_full_kernel<<<grid, kRedThreads, 0, stream>>>(pc.view(), nloc, local, loc2glob, full);
    CUADMM_CUDA(cudaGetLastError());
}

}  // namespace cuadmm

extern "C" int cuadmm_unique_id(char out[128]) {
    return cuadmm::guarded([&] { CUADMM_REQUIRE(out, "null argument"); cuadmm::make_unique_id(out); });
}
// kept for callers of the removed NCCL transport: the same job id
extern "C" int cuadmm_nccl_unique_id(char out[128]) { return cuadmm_unique_id(out); }

// ------------------------------------------------------------------------------------------
// measurement hook (not in the public header): raw cost of the cross-GPU handshakes
// ------------------------------------------------------------------------------------------
namespace cuadmm {
// mode 0: enter + leave per round (what a pushing kernel pays); mode 1: leave only; mode 2: leave only, spin on a
// volatile load without nanosleep
__global__ void peer_handshake_probe_kernel(PeerView pv, int rounds, int mode) {
    for (int i = 0; i < rounds; ++i) {
        const unsigned long long e = peer_epoch(pv);
        if (mode == 0) peer_enter(pv, e);
        if (mode == 2) {
            __syncthreads();
            if ((int)threadIdx.x < pv.world) {
                __threadfence_system();
                peer_st_release(pv.fin[threadIdx.x] + pv.rank, e);
                const volatile unsigned long long* f = pv.fin[pv.rank] + threadIdx.x;
                while (*f < e) { }
                __threadfence_system();
            }
            __syncthreads();
            if (threadIdx.x == 0) { *reinterpret_cast<volatile unsigned long long*>(pv.epoch) = e; __threadfence(); }
            __syncthreads();
        } else {
            peer_leave(pv, e);
            __syncthreads();
        }
    }
}
}  // namespace cuadmm

extern "C" int cuadmm_debug_peer_handshake(int rank, int world, const char id[128], int device, int rounds, double out_us[3]) {
    return cuadmm::guarded([&] {
        cuadmm::PeerComm pc;
        pc.init(rank, world, id, device, 1 << 16);
        cudaStream_t st;
        CUADMM_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
        cudaEvent_t e0, e1;
        CUADMM_CUDA(cudaEventCreate(&e0)); CUADMM_CUDA(cudaEventCreate(&e1));
        for (int mode = 0; mode < 3; ++mode) {
            cuadmm::peer_handshake_probe_kernel<<<1, 32, 0, st>>>(pc.view(), 10, mode);     // warm-up, aligns the ranks
            CUADMM_CUDA(cudaEventRecord(e0, st));
            cuadmm::peer_handshake_probe_kernel<<<1, 32, 0, st>>>(pc.view(), rounds, mode);
            CUADMM_CUDA(cudaEventRecord(e1, st));
            CUADMM_CUDA(cudaStreamSynchronize(st));
            float ms = 0.f;
            cudaEventElapsedTime(&ms, e0, e1);
            out_us[mode] = 1e3 * ms / rounds;
        }
        pc.check(st);
        cudaEventDestroy(e0); cudaEventDestroy(e1); cudaStreamDestroy(st);
    });
}
