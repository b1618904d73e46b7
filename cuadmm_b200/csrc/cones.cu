// cones.cu — projection onto the linear cones: 'l' blocks (nonnegative orthant, Pi(x) = max(x, 0)) and 'u' blocks
// (free variables, Pi(x) = x, dual cone {0}).  One launch covers every 'l' / 'u' entry of a plan: the blocks are cut at
// plan time into a flat list of chunks (svec offset, length, cone), one CTA per chunk.  Bandwidth-bound: per entry it
// reads Xb and writes Xproj (16 B), with the fused ADMM epilogue it also reads X, Rd1, C and writes S, S - C (56 B).
//   'l':  S = (Xproj - X) / sig - Rd1, SmC = S - C   (the arithmetic of the PSD kernels' epilogue)
//   'u':  S = 0 exactly, SmC = 0 - C                  (S lies in the dual cone {0}; not computed, so no rounding)
#include "plan.h"

namespace cuadmm {

namespace {

constexpr int kLinThreads = 256;
constexpr int kLinUnroll = 4;        // pairs in flight per thread: 4 x 16 B from each of up to 5 streams

struct LinArgs {
    const LinChunk* chunks;
    const double* __restrict__ Xb;
    double* __restrict__ Xproj;
    ProjEpilogue epi;
    const int* done_flag;
    int vec_ok;                      // every base pointer 16-byte aligned: entries 2i, 2i+1 move as one double2
};

template <bool EPI, bool FREE>
__device__ __forceinline__ void lin_one(const LinArgs& a, int64_t i, double sig) {
    const double xb = a.Xb[i];
    const double out = FREE ? xb : (xb < 0.0 ? 0.0 : xb);     // max(x, 0); NaN propagates like the PSD kernels
    a.Xproj[i] = out;
    if (EPI) {
        if (FREE) {
            a.epi.S[i] = 0.0;
            a.epi.SmC[i] = 0.0 - a.epi.Cd[i];
        } else {
            const double Sv = (out - a.epi.X[i]) / sig - a.epi.Rd1[i];
            a.epi.S[i] = Sv;
            a.epi.SmC[i] = Sv - a.epi.Cd[i];
        }
    }
}

template <bool EPI, bool FREE>
__device__ __forceinline__ void lin_chunk(const LinArgs& a, int64_t off, int len) {
    const int tid = threadIdx.x;
    const double sig = EPI && !FREE ? *a.epi.sig_ptr : 1.0;
    if (!a.vec_ok) {
        for (int e0 = tid; e0 < len; e0 += kLinThreads * kLinUnroll) {
#pragma unroll
            for (int u = 0; u < kLinUnroll; ++u) {
                const int e = e0 + u * kLinThreads;
                if (e < len) lin_one<EPI, FREE>(a, off + e, sig);
            }
        }
        return;
    }
    // an odd offset leaves one scalar entry in front of the pairs, an odd remainder one behind them
    const int head = (int)(off & 1);
    const int npairs = (len - head) >> 1;
    if (tid == 0 && head && len > 0) lin_one<EPI, FREE>(a, off, sig);
    if (tid == 1 && head + 2 * npairs < len) lin_one<EPI, FREE>(a, off + head + 2 * npairs, sig);
    const int64_t p0 = (off + head) >> 1;                    // index of the first pair in double2 units
    const double2* __restrict__ xb2 = reinterpret_cast<const double2*>(a.Xb) + p0;
    double2* __restrict__ xp2 = reinterpret_cast<double2*>(a.Xproj) + p0;
    for (int q0 = tid; q0 < npairs; q0 += kLinThreads * kLinUnroll) {
        double2 xb[kLinUnroll], x[kLinUnroll], rd[kLinUnroll], cd[kLinUnroll];
#pragma unroll
        for (int u = 0; u < kLinUnroll; ++u) {
            const int q = q0 + u * kLinThreads;
            if (q < npairs) {
                xb[u] = __ldg(xb2 + q);
                if (EPI) {
                    cd[u] = __ldg(reinterpret_cast<const double2*>(a.epi.Cd) + p0 + q);
                    if (!FREE) {
                        x[u] = __ldg(reinterpret_cast<const double2*>(a.epi.X) + p0 + q);
                        rd[u] = __ldg(reinterpret_cast<const double2*>(a.epi.Rd1) + p0 + q);
                    }
                }
            }
        }
#pragma unroll
        for (int u = 0; u < kLinUnroll; ++u) {
            const int q = q0 + u * kLinThreads;
            if (q >= npairs) continue;
            double2 out;
            out.x = FREE ? xb[u].x : (xb[u].x < 0.0 ? 0.0 : xb[u].x);
            out.y = FREE ? xb[u].y : (xb[u].y < 0.0 ? 0.0 : xb[u].y);
            xp2[q] = out;
            if (EPI) {
                double2 Sv, SmC;
                if (FREE) {
                    Sv.x = 0.0; Sv.y = 0.0;
                    SmC.x = 0.0 - cd[u].x; SmC.y = 0.0 - cd[u].y;
                } else {
                    Sv.x = (out.x - x[u].x) / sig - rd[u].x;
                    Sv.y = (out.y - x[u].y) / sig - rd[u].y;
                    SmC.x = Sv.x - cd[u].x; SmC.y = Sv.y - cd[u].y;
                }
                reinterpret_cast<double2*>(a.epi.S)[p0 + q] = Sv;
                reinterpret_cast<double2*>(a.epi.SmC)[p0 + q] = SmC;
            }
        }
    }
}

bool aligned16(const void* p) { return p == nullptr || ((uintptr_t)p & 15) == 0; }

}  // namespace

template <bool EPI>
__global__ void __launch_bounds__(kLinThreads) proj_linear_kernel(LinArgs a) {
    if (a.done_flag && *a.done_flag) return;
    const LinChunk c = a.chunks[blockIdx.x];
    if (c.cone == 'u') lin_chunk<EPI, true>(a, c.off, c.len);
    else lin_chunk<EPI, false>(a, c.off, c.len);
}

std::vector<LinChunk> linear_chunks(const BlockLayout& layout) {
    std::vector<LinChunk> out;
    const int64_t nblk = (int64_t)layout.blk.size();
    int64_t k = 0;
    while (k < nblk) {
        const char t = layout.types[k];
        if (t == 's') { ++k; continue; }
        // a run of consecutive blocks of one linear cone is one contiguous svec range
        int64_t e = k + 1;
        while (e < nblk && layout.types[e] == t) ++e;
        for (int64_t o = layout.svec_off[k]; o < layout.svec_off[e]; o += kLinearChunk) {
            LinChunk c;
            c.off = o;
            c.len = (int32_t)std::min<int64_t>(kLinearChunk, layout.svec_off[e] - o);
            c.cone = t;
            out.push_back(c);
        }
        k = e;
    }
    return out;
}

int linear_project(const LinChunk* d_chunks, int64_t nchunks, const double* Xb, double* Xproj, cudaStream_t st,
                   const ProjEpilogue* epi, const int* done_flag) {
    CUADMM_REQUIRE(nchunks <= 0x7fffffffll, "too many linear-cone chunks for one launch");
    LinArgs a;
    a.chunks = d_chunks;
    a.Xb = Xb; a.Xproj = Xproj;
    a.done_flag = done_flag;
    if (epi && epi->X) a.epi = *epi;
    else { a.epi.X = nullptr; a.epi.Rd1 = nullptr; a.epi.Cd = nullptr; a.epi.S = nullptr; a.epi.SmC = nullptr; a.epi.sig_ptr = nullptr; }
    a.vec_ok = aligned16(Xb) && aligned16(Xproj) && aligned16(a.epi.X) && aligned16(a.epi.Rd1) && aligned16(a.epi.Cd) &&
               aligned16(a.epi.S) && aligned16(a.epi.SmC);
    if (a.epi.X) proj_linear_kernel<true><<<(unsigned)nchunks, kLinThreads, 0, st>>>(a);
    else proj_linear_kernel<false><<<(unsigned)nchunks, kLinThreads, 0, st>>>(a);
    CUADMM_CUDA(cudaGetLastError());
    return 1;
}

}  // namespace cuadmm
