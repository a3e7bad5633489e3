// Device helpers shared by the Chebyshev kernels (cheb.cu: generic BSR rows, cheb_ell.cu: padded
// fixed-width rows).  Internal, not part of the ABI.
#pragma once

#include "bdg_internal.h"

namespace {

constexpr int kWarps = 4;  // 128-thread CTAs: finer occupancy granularity at ~96 registers/thread
constexpr int kThreads = kWarps * 32;
constexpr int kGroups = kThreads / 16;  // strided CTA groups in the last-CTA reduction
constexpr unsigned kFull = 0xffffffffu;

__device__ __forceinline__ void dmma_8x8x4(double &c0, double &c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

// 128-bit global loads as volatile asm: together with the (volatile) MMAs this pins the program
// order "all loads of a row, then all MMAs", which the compiler otherwise interleaves to save
// registers -- turning one HBM round trip per row into two or three.
__device__ __forceinline__ double2 ld_stream(const double2 *p) {  // read-once data (matrix blocks)
    double2 v;
    asm volatile("ld.global.cs.v2.f64 {%0,%1}, [%2];\n" : "=d"(v.x), "=d"(v.y) : "l"(p));
    return v;
}
__device__ __forceinline__ double2 ld_reuse(const double2 *p) {  // vector records (re-read by neighbours)
    double2 v;
    asm volatile("ld.global.nc.v2.f64 {%0,%1}, [%2];\n" : "=d"(v.x), "=d"(v.y) : "l"(p));
    return v;
}
__device__ __forceinline__ double2 ld_plain(const double2 *p) {
    double2 v;
    asm volatile("ld.global.v2.f64 {%0,%1}, [%2];\n" : "=d"(v.x), "=d"(v.y) : "l"(p));
    return v;
}

__device__ __forceinline__ uint64_t mix64(uint64_t z) {
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

// ---- per-step reduction of the two dot products ---------------------------------------------
// Every lane arrives with its partial sums for column `col` (valid iff col_ok and it is the
// designated leader lane for that column inside the warp).  CTA partials go to global memory;
// the last CTA of a panel to arrive adds them up in a fixed order (deterministic results) and
// writes the step's dot products.
template <int PW>
__device__ __forceinline__ void finish_dots(double d0, double d1, int col, bool leader, int panel, int n_panels,
                                            double *__restrict__ partials, unsigned *__restrict__ tickets,
                                            double *__restrict__ dots_step) {
    __shared__ double red[kWarps][2][8];
    __shared__ double comb[kGroups][16];
    __shared__ bool is_last;
    const int warp = threadIdx.x >> 5;
    if (leader) {
        red[warp][0][col] = d0;
        red[warp][1][col] = d1;
    }
    __syncthreads();
    const int which = (threadIdx.x >> 3) & 1, c = threadIdx.x & 7;
    if (threadIdx.x < 16 && c < PW) {
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) s += red[w][which][c];
        partials[((size_t)(panel * gridDim.x + blockIdx.x) * 2 + which) * 8 + c] = s;
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) is_last = atomicAdd(&tickets[panel], 1u) == gridDim.x - 1;
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    // 16 (which, column) slots x kGroups strided groups of CTAs, then a fixed-order combine.
    const int slot = threadIdx.x & 15, group = threadIdx.x >> 4;
    double s = 0.0;
    for (unsigned b = group; b < gridDim.x; b += kGroups)
        s += __ldcg(&partials[((size_t)(panel * gridDim.x + b) * 2) * 8 + slot]);
    comb[group][slot] = s;
    __syncthreads();
    if (threadIdx.x < 16 && c < PW) {
        double t = 0.0;
#pragma unroll
        for (int g = 0; g < kGroups; ++g) t += comb[g][threadIdx.x];
        dots_step[(size_t)which * n_panels * PW + panel * PW + c] = t;
    }
    if (threadIdx.x == 0) tickets[panel] = 0u;
}

}  // namespace
