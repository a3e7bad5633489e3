// Shared-memory staging helpers of the two-steps-per-pass kernels (cheb_pair.cu: one-dimensional x-planes,
// cheb_cube.cu: three-dimensional lattices): mbarriers, bulk async copies (TMA), 128-bit shared-memory accesses,
// and their reduction of the dot products.  Internal, not part of the ABI.
#pragma once

#include <stdint.h>

#include "cheb_device.cuh"

namespace {

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(bytes) : "memory");
}
// One contiguous run global -> shared through the TMA unit (SASS UBLKCP); bytes % 16 == 0.
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
    } while (!done);
}
__device__ __forceinline__ double2 lds_rec(uint32_t addr) {
    double2 v;
    asm volatile("ld.shared.v2.f64 {%0,%1}, [%2];\n" : "=d"(v.x), "=d"(v.y) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ void sts_rec(uint32_t addr, double2 v) {
    asm volatile("st.shared.v2.f64 [%0], {%1,%2};\n" ::"r"(addr), "d"(v.x), "d"(v.y) : "memory");
}

// T_{n-1}: read exactly once per launch -- do not let it displace anything in L1
__device__ __forceinline__ double2 ld_prev(const double2 *p) {
    double2 v;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0,%1}, [%2];\n" : "=d"(v.x), "=d"(v.y) : "l"(p));
    return v;
}
// ... and E_{j-1} of the T2 mode, which the same thread overwrites one iteration later (no .nc)
__device__ __forceinline__ double2 ld_prev_rw(const double2 *p) {
    double2 v;
    asm volatile("ld.global.L1::no_allocate.v2.f64 {%0,%1}, [%2];\n" : "=d"(v.x), "=d"(v.y) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void ld_table_pred(double &v, const double *p, unsigned take) {
    asm volatile("{\n .reg .pred p;\n setp.ne.u32 p, %2, 0;\n @p ld.global.nc.f64 %0, [%1];\n}\n" : "+d"(v) : "l"(p), "r"(take));
}

// Keep a value in its register: the compiler otherwise re-derives loop invariants (shared-memory
// base, lane offsets) inside the row loop, which is instruction-issue-bound.
__device__ __forceinline__ void pin(uint32_t &v) { asm volatile("" : "+r"(v)); }

// The four dot products of a run (= the pieces of one panel a CTA works through) on PW-column panels: components (quad of
// lanes) -> at PW = 4 the two sites of a warp (lane halves) -> warp -> CTA -> partials[run]; the last run of a panel to
// arrive (runs r0 .. r1) adds the panel's partials up in run order, so the result is bit-reproducible.  Called by all
// NW warps between two pieces or at the end: the rings are idle and serve as scratch.
template <int NW, int PW>
__device__ __forceinline__ void flush_dots(double d0, double d1, double d2, double d3, unsigned char *scratch, int run, int r0, int r1,
                                           int panel, int n_panels, double *__restrict__ partials, unsigned *__restrict__ tickets,
                                           double *__restrict__ dots_step) {
    static_assert(PW == 4 || PW == 8, "a lane holds one (column, component) element of one site");
    constexpr int N = 4 * PW;  // slots: which * PW + column; which = (step within the pair) * 2 + (0: <T,T>, 1: <T',T>)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __shared__ bool is_last;
    d0 += __shfl_xor_sync(kFull, d0, 1);
    d1 += __shfl_xor_sync(kFull, d1, 1);
    d2 += __shfl_xor_sync(kFull, d2, 1);
    d3 += __shfl_xor_sync(kFull, d3, 1);
    d0 += __shfl_xor_sync(kFull, d0, 2);
    d1 += __shfl_xor_sync(kFull, d1, 2);
    d2 += __shfl_xor_sync(kFull, d2, 2);
    d3 += __shfl_xor_sync(kFull, d3, 2);
    if (PW == 4) {
        d0 += __shfl_xor_sync(kFull, d0, 16);
        d1 += __shfl_xor_sync(kFull, d1, 16);
        d2 += __shfl_xor_sync(kFull, d2, 16);
        d3 += __shfl_xor_sync(kFull, d3, 16);
    }
    __syncthreads();
    double *red = reinterpret_cast<double *>(scratch);  // [NW][4 which][PW columns], then comb [NW][N] behind it
    double *comb = red + NW * N;
    if ((PW == 8 || lane < 16) && (lane & 3) == 0) {
        const int col = lane >> 2;
        red[(warp * 4 + 0) * PW + col] = d0;
        red[(warp * 4 + 1) * PW + col] = d1;
        red[(warp * 4 + 2) * PW + col] = d2;
        red[(warp * 4 + 3) * PW + col] = d3;
    }
    __syncthreads();
    if (threadIdx.x < N) {
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < NW; ++w) s += red[w * N + threadIdx.x];
        partials[(size_t)run * N + threadIdx.x] = s;
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) is_last = atomicAdd(&tickets[panel], 1u) == (unsigned)(r1 - r0 - 1);
    __syncthreads();
    if (is_last) {
        __threadfence();
        if (PW == 8 || lane < 16) {
            double s = 0.0;
            for (int b = r0 + warp; b < r1; b += NW) s += __ldcg(&partials[(size_t)b * N + lane]);
            comb[warp * N + lane] = s;
        }
        __syncthreads();
        if (threadIdx.x < N) {
            double t = 0.0;
#pragma unroll
            for (int g = 0; g < NW; ++g) t += comb[g * N + threadIdx.x];
            dots_step[(size_t)(threadIdx.x / PW) * n_panels * PW + panel * PW + (threadIdx.x % PW)] = t;
        }
        if (threadIdx.x == 0) tickets[panel] = 0u;
    }
    __syncthreads();  // scratch and is_last are free again
}

}  // namespace
