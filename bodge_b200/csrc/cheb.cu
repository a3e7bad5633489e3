// Chebyshev / kernel-polynomial engine: fused block-sparse SpMM + three-term update + moment
// dot products, one HBM pass per step.
//
//   T_{n+1} = alpha * H * T_n - beta * T_{n-1}      (alpha = 2/a, beta = 1;  first step: 1/a, 0)
//   d0 = <T_n, T_n>,  d1 = <T_{n+1}, T_n>           (per column; give mu_2n and mu_2n+1)
//
// There is no reference code for this (SURVEY 0.2); the arithmetic it must reproduce is scipy's
// bsr_matvecs on the reference's matrix("bsr") driven by the textbook recursion (oracle/).
//
// Data layout in HBM
//   matrix : the compacted BSR exactly as exported (indptr int32, indices int32, data [nb][4][4]
//            complex128, 256 B per block, row-major inside the block).
//   vectors: column panels of PW in {1,2,4,8} columns; inside a panel one contiguous record per
//            site, [site][column][alpha] complex128 = 64*PW bytes (512 B at PW = 8).  A warp
//            reads or writes a whole record with one 128-bit access per lane.
//
// Kernel (cheb_step_dmma): one warp per block row.  The 4x4 complex block times the 4xPW complex
// record is the real product [[Br,-Bi],[Bi,Br]] (8x8) x [Xr;Xi] (8xPW): exactly two FP64
// m8n8k4 warp-level MMAs, with lane l fetching block element l%16 and record element l -- both
// fully coalesced, no shared-memory staging, ~40 registers, so 64 resident warps per SM hide the
// HBM latency by thread-level parallelism.  The kernel is bandwidth-bound; the MMA form is used
// because it removes the FP64 issue/broadcast overhead a scalar formulation has (SURVEY H3), not
// to chase flops.  cheb_step_fma is the scalar-FMA formulation of the same step (A/B reference).
#include <algorithm>
#include <cstring>

#include "bdg_internal.h"
#include "cheb_device.cuh"
#include "cheb_plan.h"

namespace {

// ---- the fused step: FP64 warp-MMA formulation --------------------------------------------------
// CH = neighbour blocks handled per round; the host picks the smallest instantiated CH that
// covers the longest block row (5 for 2-D lattices, 7 for 3-D), so a row is ONE round:
//   1. consume what earlier iterations prefetched (this row's block range and block columns),
//   2. issue every load of the row back to back -- CH blocks, CH neighbour records, T_n and
//      T_{n-1} of the row itself, and the index prefetches for the next rows,
//   3. 2*CH MMAs, re/im exchange, update, dots, one store.
// Straight-line code: slots past the end of a short row load a valid dummy address and feed
// zeros to the MMA (no divergence handling, and no scoreboard slot shared between data that is
// consumed now and loads that were issued just before -- the SASS has only six).
template <int PW, bool FIRST, int CH>
__global__ void __launch_bounds__(kThreads, 4)
cheb_step_dmma(const int32_t *__restrict__ indptr, const int32_t *__restrict__ indices,
               const double2 *__restrict__ data, const double2 *__restrict__ x_cur, double2 *__restrict__ x_io,
               int n_sites, double alpha, double beta, double *__restrict__ partials,
               unsigned *__restrict__ tickets, double *__restrict__ dots_step, int n_panels) {
    constexpr int REC = PW * 4;  // complex elements per site record
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int panel = blockIdx.y;
    const double2 *__restrict__ xc = x_cur + (size_t)panel * n_sites * REC;
    double2 *__restrict__ xo = x_io + (size_t)panel * n_sites * REC;
    // Row traversal: the whole grid sweeps the lattice as one wavefront -- in pass t, CTA b works on
    // rows (t * gridDim.x + b) * kWarps ... + kWarps - 1.  All SMs then touch one window of a few
    // thousand consecutive sites at a time, so the records of the +-Ly / +-LyLz neighbours (read
    // again one or two passes later) are still in L2 and every vector byte leaves HBM once.
    const int stride = gridDim.x * kWarps;

    // A-operand role: lanes 0-15 feed rows 0-3 of [[Br,-Bi],[Bi,Br]], lanes 16-31 rows 4-7.
    const int elem = lane & 15;
    const bool hi = lane >= 16;
    // B-operand role: lane l holds record element l = (column l/4, alpha l%4); lanes past the
    // record (PW < 8) read element 0 and contribute zeros.
    const bool x_lane = lane < REC;
    const int x_elem = x_lane ? lane : 0;
    // Output role after the re/im exchange: lane owns T_{n+1}[row][alpha=a][column=col].
    const int a = (lane >> 2) & 3;
    const int col = 2 * (lane & 3) + (lane >> 4);
    const bool o_lane = col < PW;
    const int o_elem = o_lane ? col * 4 + a : 0;

    int row = blockIdx.x * kWarps + warp;
    int p0 = 0, p1 = 0, q0 = 0, q1 = 0, jv = 0;  // [p0,p1): this row's blocks, [q0,q1): next row's
    if (row < n_sites) {
        p0 = __ldg(indptr + row);
        p1 = __ldg(indptr + row + 1);
    }
    if (row + stride < n_sites) {
        q0 = __ldg(indptr + row + stride);
        q1 = __ldg(indptr + row + stride + 1);
    }
    if (lane < p1 - p0) jv = __ldg(indices + p0 + lane);

    double d0 = 0.0, d1 = 0.0;
    for (; row < n_sites; row += stride) {
        // (1) consume prefetched index data: neighbour ids of the first CH blocks
        const int cnt = p1 - p0;
        int jn_u[CH];
#pragma unroll
        for (int u = 0; u < CH; ++u) {
            const int j = __shfl_sync(kFull, jv, u);
            jn_u[u] = u < cnt ? j : row;  // dummy: the row's own record (always valid)
        }
        // (2) all loads of the row
        double2 bv[CH], xv[CH];
#pragma unroll
        for (int u = 0; u < CH; ++u) {
            const int p = u < cnt ? p0 + u : p0;
            bv[u] = ld_stream(data + (size_t)p * 16 + elem);
            xv[u] = ld_reuse(xc + (size_t)jn_u[u] * REC + x_elem);
        }
        const size_t off = (size_t)row * REC + o_elem;
        const double2 tn = ld_reuse(xc + off);
        double2 pv = make_double2(0.0, 0.0);
        if (!FIRST) pv = ld_plain(xo + off);
        int r0 = 0, r1 = 0, jn = 0;
        if (row + 2 * stride < n_sites) {
            r0 = __ldg(indptr + row + 2 * stride);
            r1 = __ldg(indptr + row + 2 * stride + 1);
        }
        if (lane < q1 - q0) jn = __ldg(indices + q0 + lane);

        // (3) MMAs: two independent accumulation chains
        double re0 = 0.0, re1 = 0.0, im0 = 0.0, im1 = 0.0;
#pragma unroll
        for (int u = 0; u < CH; ++u) {
            const bool live = u < cnt;
            const double xr = (live && x_lane) ? xv[u].x : 0.0;
            const double xi = (live && x_lane) ? xv[u].y : 0.0;
            dmma_8x8x4(re0, re1, hi ? bv[u].y : bv[u].x, xr);   // [Br; Bi]  * Xr
            dmma_8x8x4(im0, im1, hi ? bv[u].x : -bv[u].y, xi);  // [-Bi; Br] * Xi
        }
        // rows longer than CH blocks (generic lattices): plain loop over the rest
        for (int t = CH; t < cnt; ++t) {
            const int j = __ldg(indices + p0 + t);
            const double2 b2 = __ldcs(data + (size_t)(p0 + t) * 16 + elem);
            const double2 x2 = __ldg(xc + (size_t)j * REC + x_elem);
            dmma_8x8x4(re0, re1, hi ? b2.y : b2.x, x_lane ? x2.x : 0.0);
            dmma_8x8x4(im0, im1, hi ? b2.x : -b2.y, x_lane ? x2.y : 0.0);
        }
        const double c0 = re0 + im0, c1 = re1 + im1;
        // Lanes < 16 hold Re(y) of (a, columns 2q, 2q+1), lanes >= 16 the matching Im(y):
        // swap one value with the partner lane so each lane owns one complex element.
        const double recv = __shfl_xor_sync(kFull, hi ? c0 : c1, 16);
        const double yr = hi ? recv : c0;
        const double yi = hi ? c1 : recv;
        if (o_lane) {
            const double2 out = make_double2(alpha * yr - beta * pv.x, alpha * yi - beta * pv.y);
            xo[off] = out;
            d0 += tn.x * tn.x + tn.y * tn.y;
            d1 += out.x * tn.x + out.y * tn.y;
        }
        p0 = q0; p1 = q1; jv = jn;
        q0 = r0; q1 = r1;
    }
    // lanes sharing a column differ in alpha (lane bits 2,3)
    d0 += __shfl_xor_sync(kFull, d0, 4);
    d1 += __shfl_xor_sync(kFull, d1, 4);
    d0 += __shfl_xor_sync(kFull, d0, 8);
    d1 += __shfl_xor_sync(kFull, d1, 8);
    finish_dots<PW>(d0, d1, col, o_lane && a == 0, panel, n_panels, partials, tickets, dots_step);
}

// ---- the fused step: scalar FMA formulation (one thread per (site, column)) ----------------------
template <int PW, bool FIRST>
__global__ void __launch_bounds__(kThreads)
cheb_step_fma(const int32_t *__restrict__ indptr, const int32_t *__restrict__ indices,
              const double2 *__restrict__ data, const double2 *__restrict__ x_cur, double2 *__restrict__ x_io,
              int n_sites, double alpha, double beta, double *__restrict__ partials,
              unsigned *__restrict__ tickets, double *__restrict__ dots_step, int n_panels) {
    constexpr int REC = PW * 4;
    constexpr int ROWS_PER_WARP = 32 / PW;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int panel = blockIdx.y;
    const double2 *__restrict__ xc = x_cur + (size_t)panel * n_sites * REC;
    double2 *__restrict__ xo = x_io + (size_t)panel * n_sites * REC;
    // same wavefront traversal as cheb_step_dmma
    const int col = lane % PW, sub = lane / PW;

    double d0 = 0.0, d1 = 0.0;
    for (int base = (blockIdx.x * kWarps + warp) * ROWS_PER_WARP; base < n_sites;
         base += gridDim.x * kWarps * ROWS_PER_WARP) {
        const int row = base + sub;
        if (row >= n_sites) continue;
        double2 acc[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) acc[r] = make_double2(0.0, 0.0);
        for (int p = indptr[row]; p < indptr[row + 1]; ++p) {
            const int j = indices[p];
            const double2 *xb = xc + (size_t)j * REC + col * 4;
            const double2 *blk = data + (size_t)p * 16;
            double2 x[4];
#pragma unroll
            for (int b = 0; b < 4; ++b) x[b] = __ldg(xb + b);
#pragma unroll
            for (int r = 0; r < 4; ++r) {
#pragma unroll
                for (int b = 0; b < 4; ++b) {
                    const double2 m = __ldg(blk + r * 4 + b);
                    acc[r].x += m.x * x[b].x - m.y * x[b].y;
                    acc[r].y += m.x * x[b].y + m.y * x[b].x;
                }
            }
        }
        const size_t off = (size_t)row * REC + col * 4;
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const double2 tn = __ldg(xc + off + r);
            double2 out;
            if (FIRST) {
                out = make_double2(alpha * acc[r].x, alpha * acc[r].y);
            } else {
                const double2 pv = xo[off + r];
                out = make_double2(alpha * acc[r].x - beta * pv.x, alpha * acc[r].y - beta * pv.y);
            }
            xo[off + r] = out;
            d0 += tn.x * tn.x + tn.y * tn.y;
            d1 += out.x * tn.x + out.y * tn.y;
        }
    }
#pragma unroll
    for (int d = PW; d < 32; d <<= 1) {
        d0 += __shfl_xor_sync(kFull, d0, d);
        d1 += __shfl_xor_sync(kFull, d1, d);
    }
    finish_dots<PW>(d0, d1, col, sub == 0, panel, n_panels, partials, tickets, dots_step);
}

// ---- start vectors ----------------------------------------------------------------------------
// One thread per complex element of the padded vector set; columns >= n_cols are zero.
__global__ void __launch_bounds__(kThreads)
init_rademacher(double2 *__restrict__ x, int64_t n_elems, int n_sites, int pw, int n_cols, uint64_t seed,
                int64_t col_offset) {
    int64_t t = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (t >= n_elems) return;
    const int alpha = (int)(t & 3);
    const int c = (int)((t >> 2) % pw);
    const int64_t rec = (t >> 2) / pw;
    const int site = (int)(rec % n_sites);
    const int panel = (int)(rec / n_sites);
    const int colg = panel * pw + c;
    double v = 0.0;
    if (colg < n_cols) {
        const uint64_t G = 0x9E3779B97F4A7C15ull;
        const uint64_t hc = mix64(seed + G * ((uint64_t)(col_offset + colg) + 1ull));
        const uint64_t h = mix64(hc + G * ((uint64_t)(4 * (int64_t)site + alpha) + 1ull));
        v = (h >> 63) ? -1.0 : 1.0;
    }
    x[t] = make_double2(v, 0.0);
}

// Class columns: column c is the indicator of class class_rows[c] >> 2 in component class_rows[c] & 3.  One thread per
// complex element of the padded vector set, like init_rademacher.
__global__ void __launch_bounds__(kThreads)
init_classes(double2 *__restrict__ x, int64_t n_elems, int n_sites, int pw, int n_cols, const int32_t *__restrict__ site_class,
             const int64_t *__restrict__ class_rows) {
    int64_t t = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (t >= n_elems) return;
    const int alpha = (int)(t & 3);
    const int c = (int)((t >> 2) % pw);
    const int64_t rec = (t >> 2) / pw;
    const int site = (int)(rec % n_sites);
    const int panel = (int)(rec / n_sites);
    const int colg = panel * pw + c;
    double v = 0.0;
    if (colg < n_cols) {
        const int64_t q = class_rows[colg];
        v = (alpha == (int)(q & 3) && (int64_t)site_class[site] == (q >> 2)) ? 1.0 : 0.0;
    }
    x[t] = make_double2(v, 0.0);
}

__global__ void init_probes(double2 *__restrict__ x, int n_sites, int pw, int n_cols,
                            const int64_t *__restrict__ probe_rows) {
    int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_cols) return;
    const int64_t r = probe_rows[c];
    const int64_t site = r >> 2;
    const int alpha = (int)(r & 3);
    const int panel = c / pw, cl = c % pw;
    x[(((size_t)panel * n_sites + site) * pw + cl) * 4 + alpha] = make_double2(1.0, 0.0);
}

// T2 mode: the launches leave rows (a_j, c_j, b_j, d_j) = (<E_j,E_j>, <u_j,E_j>, <E_{j+1},E_j>, <E_{j+1},u_j>) with
// E_j = T_2j x, u_j = H~ E_j.  From T_m T_n = (T_{m+n} + T_|m-n|) / 2:
//     a_j = (mu_4j + mu_0)/2,                      b_j = (mu_{4j+2} + mu_2)/2,
//     c_j = (mu_{4j+1} + mu_{4j-1})/4 + mu_1/2,    d_j = (mu_{4j+3} + mu_{4j+1})/4 + (mu_3 + mu_1)/4.
// This rewrites the rows as the single-step kernels would have left them, D_n = (mu_n + mu_{n mod 2})/2, so that
// every consumer (moments_from_dots, observables.cu) reads one format.  One thread per column; the odd moments
// are a two-term recurrence along j.  Measured against an extended-precision recursion (tests/test_gpu_readout.py), their
// worst error on a 6 x 5 open plane is 0.33, 2.1 and 3.5 x (n+1) eps mu_0 at 2048, 32768 and 131072 moments (DESIGN 4.1).
__global__ void __launch_bounds__(kThreads)
t2_normalize(double *__restrict__ dots, int stride, int j_begin, int j_end) {
    const int c = blockIdx.x * kThreads + threadIdx.x;
    if (c >= stride) return;
    auto row = [&](int n) -> double & { return dots[(size_t)n * stride + c]; };
    if (j_begin == 0) {  // mu_0 = a_0, mu_1 = c_0, mu_2 = b_0, (mu_3 + mu_1)/2 = d_0
        row(2) = 0.5 * (row(2) + row(0));
        j_begin = 1;
    }
    const double mu0 = row(0), mu1 = row(1), mu2 = 2.0 * row(2) - mu0, mu3 = 2.0 * row(3) - mu1;
    double odd = 2.0 * row(4 * j_begin - 1) - mu1;  // mu_{4j-1}
    // Chunks of kChunk launches: all loads of a chunk are issued before its first store (the stores go to the
    // same array, so the compiler cannot hoist later loads over them: one memory latency per chunk, not per j).
    constexpr int kChunk = 8;
    for (int j0 = j_begin; j0 < j_end; j0 += kChunk) {
        double cj[kChunk], bj[kChunk], dj[kChunk];
#pragma unroll
        for (int i = 0; i < kChunk; ++i) {
            const int j = min(j0 + i, j_end - 1);
            cj[i] = row(4 * j + 1), bj[i] = row(4 * j + 2), dj[i] = row(4 * j + 3);
        }
#pragma unroll
        for (int i = 0; i < kChunk; ++i) {
            const int j = j0 + i;
            if (j < j_end) {
                const double m1 = 4.0 * cj[i] - 2.0 * mu1 - odd;   // mu_{4j+1}
                const double m3 = 4.0 * dj[i] - (mu3 + mu1) - m1;  // mu_{4j+3}
                row(4 * j + 1) = 0.5 * (m1 + mu1);
                row(4 * j + 2) = bj[i] - 0.5 * mu2 + 0.5 * mu0;
                row(4 * j + 3) = 0.5 * (m3 + mu1);
                odd = m3;
            }
        }
    }
}

// mu[n][c] from the per-step dot products: step s gave d0 = <T_s,T_s> (s = 0: <T_0,T_0>) and
// d1 = <T_{s+1},T_s>;  mu_{2s} = 2 d0 - mu_0, mu_{2s+1} = 2 d1 - mu_1 for s >= 1.  The flat index runs over
// n_moments * n_cols, which passes 2^31 for long per-column reads of many columns: 64-bit.
__global__ void __launch_bounds__(kThreads)
moments_from_dots(const double *__restrict__ dots, int n_moments, int n_cols, int stride /* n_panels*PW */,
                  int reduce, double *__restrict__ mu) {
    const int64_t t = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    const int64_t n_out = reduce ? 1 : n_cols;
    if (t >= (int64_t)n_moments * n_out) return;
    const int64_t n = t / n_out, c_first = reduce ? 0 : t % n_out, c_last = reduce ? n_cols : c_first + 1;
    const int64_t s = n >> 1, which = n & 1;
    double sum = 0.0;
    for (int64_t c = c_first; c < c_last; ++c) {
        const double d = dots[((size_t)s * 2 + which) * stride + c];
        sum += s == 0 ? d : 2.0 * d - dots[(size_t)which * stride + c];
    }
    mu[t] = sum;
}

// [panel][site][col][alpha] -> row-major [4N][n_cols]
__global__ void __launch_bounds__(kThreads)
unpack_vectors(const double2 *__restrict__ x, int n_sites, int pw, int n_cols, double2 *__restrict__ out) {
    int64_t t = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (t >= (int64_t)n_sites * 4 * n_cols) return;
    const int c = (int)(t % n_cols);
    const int64_t r = t / n_cols;
    const int64_t site = r >> 2;
    const int alpha = (int)(r & 3);
    out[t] = x[(((size_t)(c / pw) * n_sites + site) * pw + (c % pw)) * 4 + alpha];
}

template <int PW> StepKernel pick_pw(int kernel, bool first, int max_row) {
    if (kernel == BDG_KERNEL_FMA) return first ? cheb_step_fma<PW, true> : cheb_step_fma<PW, false>;
    if (max_row <= 3) return first ? cheb_step_dmma<PW, true, 3> : cheb_step_dmma<PW, false, 3>;
    if (max_row <= 5) return first ? cheb_step_dmma<PW, true, 5> : cheb_step_dmma<PW, false, 5>;
    if (max_row <= 7) return first ? cheb_step_dmma<PW, true, 7> : cheb_step_dmma<PW, false, 7>;
    return first ? cheb_step_dmma<PW, true, 8> : cheb_step_dmma<PW, false, 8>;
}

StepKernel pick_kernel(int kernel, int pw, bool first, int max_row) {
    switch (pw) {
        case 1: return pick_pw<1>(kernel, first, max_row);
        case 2: return pick_pw<2>(kernel, first, max_row);
        case 4: return pick_pw<4>(kernel, first, max_row);
        default: return pick_pw<8>(kernel, first, max_row);
    }
}

bool ell_format(int kernel) { return kernel == BDG_KERNEL_ELL || kernel == BDG_KERNEL_DICT || kernel == BDG_KERNEL_DICT_DIAG; }

// DMMA / FMA: the FIRST and the next-step kernel on one grid -- enough CTAs to fill every SM at the kernel's occupancy, split
// over panels; each CTA walks one contiguous range of block rows (neighbouring rows share their X records in L1).
int bsr_configure(bdg_system *sys) {
    ChebState &st = sys->cheb;
    const StepKernel next = pick_kernel(st.kernel, st.panel_width, false, sys->packed_max_row);
    int per_sm = 1;
    BDG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, next, kThreads, 0));
    per_sm = std::max(per_sm, 1);
    const int64_t target = (int64_t)sys->sm_count * per_sm;
    int64_t gx = std::max<int64_t>(1, target / st.n_panels);
    const int rows_per_warp_pass = st.kernel == BDG_KERNEL_FMA ? kWarps * (32 / st.panel_width) : kWarps;
    gx = std::min<int64_t>(gx, ceil_div(sys->packed.n_sites, rows_per_warp_pass));
    const dim3 grid((unsigned)gx, (unsigned)st.n_panels);
    st.bsr_first = {pick_kernel(st.kernel, st.panel_width, true, sys->packed_max_row), grid, kThreads, 0};
    st.bsr_next = {next, grid, kThreads, 0};
    st.partial_runs = std::max(st.partial_runs, (int)gx);
    return BDG_OK;
}

int bsr_launch(bdg_system *sys, bool first, const void *x_cur, void *x_io, double *dots_step) {
    ChebState &st = sys->cheb;
    const BsrDev &m = sys->packed;
    const Launch<StepKernel> &l = first ? st.bsr_first : st.bsr_next;
    note_launch(st, reinterpret_cast<const void *>(l.fn));
    l.fn<<<l.grid, l.threads, l.smem, sys->stream>>>(m.indptr.as<int32_t>(), m.indices.as<int32_t>(), m.data.as<double2>(),
                                                     static_cast<const double2 *>(x_cur), static_cast<double2 *>(x_io),
                                                     (int)m.n_sites, (first ? 1.0 : 2.0) / st.scale, first ? 0.0 : 1.0,
                                                     st.partials.as<double>(), st.tickets.as<unsigned>(), dots_step, st.n_panels);
    BDG_CUDA(cudaGetLastError());
    return BDG_OK;
}

int ensure_dot_capacity(bdg_system *sys, int steps_total) {
    ChebState &st = sys->cheb;
    if (steps_total + 1 <= st.dot_capacity) return BDG_OK;
    const int stride = st.n_panels * st.panel_width;
    int cap = std::max(steps_total + 1, std::max(1024, st.dot_capacity * 2));
    DevBuf grown;
    BDG_TRY(dev_alloc(sys, grown, (size_t)cap * 2 * stride * sizeof(double)));
    if (st.dots.ptr && st.dot_capacity > 0) {
        BDG_CUDA(cudaMemcpyAsync(grown.ptr, st.dots.ptr, (size_t)st.dot_capacity * 2 * stride * sizeof(double),
                                 cudaMemcpyDeviceToDevice, sys->stream));
        BDG_CUDA(cudaStreamSynchronize(sys->stream));
    }
    dev_free(sys, st.dots);
    st.dots = grown;
    st.dot_capacity = cap;
    return BDG_OK;
}

// One launch of the plan.  `first`: the launch of bdg_cheb_begin, T_1 = H~ T_0 (E_1 = T_2(H~) E_0 on the even-vector
// steppings); `remaining`: the steps still asked for, of which Pair takes two per launch while two remain (T_1 and an odd
// leftover run on its single-step kernel).  Even steppings always take two: an odd request is rounded up.
int advance(bdg_system *sys, bool first, int remaining) {
    ChebState &st = sys->cheb;
    const bool pair = st.stepping == Stepping::Pair && !first && remaining >= 2;
    if (st.even()) BDG_TRY(ensure_dot_capacity(sys, st.steps_done + 2));
    // the dot rows of step `slot` (and slot + 1 on a two-step launch): step n = steps_done + 1 when T_n is current, 0 first
    const int slot = first ? 0 : st.steps_done + 1;
    double *dots_step = st.dots.as<double>() + (size_t)slot * 2 * st.n_panels * st.panel_width;
    const void *x_cur = st.vec[st.cur].ptr;
    void *x_io = st.vec[st.prev].ptr;
    // (prev, cur) after the launch: T_{n+1} (E_{j+1}) is written over T_{n-1} (E_{j-1}); the pair kernel writes T_{n+1}, T_{n+2}
    // into the two buffers holding neither T_n nor T_{n-1}.
    int next[2] = {st.cur, st.prev};
    if (pair)
        for (int b = 0, k = 0; b < 4; ++b)
            if (b != st.cur && b != st.prev) next[k++] = b;
    switch (st.stepping) {
        case Stepping::EvenPlane: BDG_TRY(t2_launch(sys, first, x_cur, x_io, dots_step)); break;
        case Stepping::EvenCube: BDG_TRY(cube_launch(sys, first, x_cur, x_io, dots_step)); break;
        case Stepping::Pair:
            if (pair) {
                BDG_TRY(pair_launch(sys, x_io, x_cur, st.vec[next[0]].ptr, st.vec[next[1]].ptr, dots_step));
                break;
            }
            [[fallthrough]];
        case Stepping::Single:
            BDG_TRY(ell_format(st.kernel) ? ell_launch_step(sys, first, x_cur, x_io, dots_step)
                                          : bsr_launch(sys, first, x_cur, x_io, dots_step));
            break;
    }
    st.prev = next[0];
    st.cur = next[1];
    st.launches += 1;
    // the new vectors, T_{slot+1} (and T_{slot+2}), into the local accumulator; the even-vector recursion keeps every second
    // vector only and takes none (bdg_cheb_local_begin)
    if (!st.even()) BDG_TRY(local_accumulate(sys, slot + 1, st.vec[next[pair ? 0 : 1]].ptr, pair ? st.vec[next[1]].ptr : nullptr));
    st.steps_done += (pair || st.even() ? 2 : 1) - (first ? 1 : 0);
    return BDG_OK;
}

}  // namespace

// T2 mode: bring the dot rows written since the last call into the single-step format (t2_normalize).
int t2_finish_dots(bdg_system *sys) {
    ChebState &st = sys->cheb;
    if (!st.even() || !st.active) return BDG_OK;
    const int launches = (st.steps_done + 1) / 2;  // rows = 2 (steps_done + 1) = 4 per launch
    if (st.t2_rows_normalized >= launches) return BDG_OK;
    const int stride = st.n_panels * st.panel_width;
    t2_normalize<<<(unsigned)ceil_div(stride, kThreads), kThreads, 0, sys->stream>>>(st.dots.as<double>(), stride,
                                                                                     st.t2_rows_normalized, launches);
    BDG_CUDA(cudaGetLastError());
    st.t2_rows_normalized = launches;
    st.launches += 1;
    return BDG_OK;
}

void cheb_deactivate(bdg_system *sys) {
    sys->cheb.active = false;
    sys->ell.valid = false;
}

void cheb_release(bdg_system *sys) {
    ChebState &st = sys->cheb;
    cudaStreamSynchronize(sys->stream);
    for (DevBuf &v : st.vec) dev_free(sys, v);
    dev_free(sys, st.dots);
    dev_free(sys, st.partials);
    dev_free(sys, st.tickets);
    dev_free(sys, st.mu_tmp);
    dev_free(sys, st.obs_tmp);
    dev_free(sys, st.work_items);
    dev_free(sys, st.local_off);
    dev_free(sys, st.local_acc);
    ell_release(sys);
    const int64_t launches = st.launches;
    st = ChebState();
    st.launches = launches;
}

extern "C" int bdg_set_classes(bdg_t *sys, int64_t n_sites, const int32_t *site_class, int32_t n_classes) {
    BDG_ENTER(sys);
    BDG_REQUIRE(n_sites == sys->skel.n_sites, "%lld site classes given for %lld sites", (long long)n_sites,
                (long long)sys->skel.n_sites);
    BDG_REQUIRE(n_classes >= 1, "need at least one class, %d given", n_classes);
    BDG_REQUIRE(site_class != nullptr, "null argument");
    for (int64_t i = 0; i < n_sites; ++i)
        BDG_REQUIRE(site_class[i] >= 0 && site_class[i] < n_classes, "site %lld: class %d outside [0, %d)", (long long)i,
                    site_class[i], n_classes);
    sys->n_classes = 0;  // (no classes while the upload may fail half way)
    BDG_TRY(dev_alloc(sys, sys->site_class, (size_t)n_sites * sizeof(int32_t)));
    BDG_CUDA(cudaMemcpyAsync(sys->site_class.ptr, site_class, (size_t)n_sites * sizeof(int32_t), cudaMemcpyHostToDevice,
                             sys->stream));
    BDG_CUDA(cudaStreamSynchronize(sys->stream));  // site_class is borrowed only for this call
    sys->n_classes = n_classes;
    return BDG_OK;
}

extern "C" int bdg_cheb_begin(bdg_t *sys, int kind, int32_t n_cols, const int64_t *probe_rows, uint64_t seed,
                              int64_t col_offset, double scale, int kernel) {
    BDG_ENTER(sys);
    BDG_REQUIRE(kind == BDG_X0_PROBE || kind == BDG_X0_RADEMACHER || kind == BDG_X0_CLASS, "unknown start-vector kind %d", kind);
    BDG_REQUIRE(n_cols >= 1, "need at least one column");
    BDG_REQUIRE(scale > 0.0, "scale must be positive");
    BDG_REQUIRE(kind == BDG_X0_RADEMACHER || probe_rows != nullptr, kind == BDG_X0_CLASS ? "class rows missing" : "probe rows missing");
    if (kind == BDG_X0_CLASS) {
        BDG_REQUIRE(sys->n_classes > 0, "no site classes uploaded (bdg_set_classes)");
        for (int c = 0; c < n_cols; ++c)
            BDG_REQUIRE(probe_rows[c] >= 0 && (probe_rows[c] >> 2) < sys->n_classes,
                        "column %d: class row %lld names class %lld, beta %lld; classes are 0 .. %d", c, (long long)probe_rows[c],
                        (long long)(probe_rows[c] >> 2), (long long)(probe_rows[c] & 3), sys->n_classes - 1);
    }
    BDG_REQUIRE(kernel >= BDG_KERNEL_AUTO && kernel <= BDG_KERNEL_AUTO_MOMENTS && kernel != 4 && kernel != 5,  // 4, 5: unassigned (bdg.h)
                "unknown kernel %d", kernel);
    BDG_TRY(build_packed(sys));
    const PlanSwitches sw = read_plan_switches();
    PlanFacts facts{};
    if (kernel != BDG_KERNEL_DMMA && kernel != BDG_KERNEL_FMA) {  // every other kernel reads the copies of formats.cu
        BDG_TRY(ell_build(sys));
        const EllDev &e = sys->ell;
        facts = {e.usable, e.dict_usable, e.diag_usable, e.pair_usable, e.cube_usable, e.n_sites, sys->cubic[1], sys->cubic[2],
                 sys->sm_count};
    }
    const SteppingPlan plan = plan_stepping(kernel, n_cols, facts, sw);
    BDG_REQUIRE(!plan.refusal, "%s", plan.refusal);
    const BsrDev &m = sys->packed;
    const int n = (int)m.n_sites;
    if (kind == BDG_X0_PROBE)
        for (int c = 0; c < n_cols; ++c)
            BDG_REQUIRE(probe_rows[c] >= 0 && probe_rows[c] < 4 * (int64_t)n, "probe row %lld out of range", (long long)probe_rows[c]);

    // Buffers of a previous recursion are kept and reused when large enough (parameter sweeps).
    ChebState &st = sys->cheb;
    st.active = false;
    st.kernel = plan.format;
    st.n_cols = n_cols;
    st.stepping = plan.stepping;
    st.panel_width = plan.panel_width;
    st.n_panels = plan.n_panels;
    st.scale = scale;
    st.steps_done = 0;
    st.cur = 0;
    st.prev = 1;
    st.t2_rows_normalized = 0;
    st.local = false;
    st.launched.clear();
    st.last_launched = nullptr;
    st.dot_capacity = (int)(st.dots.bytes / ((size_t)2 * st.n_panels * st.panel_width * sizeof(double)));

    // The kernels the recursion will launch: the single-step kernel (every step, or T_1 and odd leftovers of the pair
    // plan), the two-step kernel, or the even-vector one.
    st.partial_runs = 0;
    if (st.stepping == Stepping::Single || st.stepping == Stepping::Pair)
        BDG_TRY(ell_format(st.kernel) ? ell_configure(sys, sw) : bsr_configure(sys));
    if (st.stepping == Stepping::Pair || st.stepping == Stepping::EvenPlane) BDG_TRY(pair_configure(sys, sw));
    if (st.stepping == Stepping::EvenCube) BDG_TRY(cube_configure(sys, sw));

    const size_t vec_elems = (size_t)st.n_panels * n * st.panel_width * 4;
    for (int b = 0; b < (st.stepping == Stepping::Pair ? 4 : 2); ++b) BDG_TRY(dev_alloc(sys, st.vec[b], vec_elems * sizeof(double2)));
    BDG_TRY(dev_alloc(sys, st.partials,
                      (size_t)st.n_panels * st.partial_runs * (st.stepping == Stepping::Single ? 16 : 32) * sizeof(double)));
    BDG_TRY(dev_alloc(sys, st.tickets, (size_t)st.n_panels * sizeof(unsigned)));
    BDG_CUDA(cudaMemsetAsync(st.tickets.ptr, 0, (size_t)st.n_panels * sizeof(unsigned), sys->stream));
    BDG_TRY(ensure_dot_capacity(sys, 1024));
    st.active = true;

    double2 *x0 = st.vec[0].as<double2>();
    if (kind == BDG_X0_RADEMACHER) {
        init_rademacher<<<(unsigned)ceil_div((int64_t)vec_elems, kThreads), kThreads, 0, sys->stream>>>(
            x0, (int64_t)vec_elems, n, st.panel_width, n_cols, seed, col_offset);
    } else if (kind == BDG_X0_CLASS) {
        BDG_TRY(dev_alloc(sys, st.mu_tmp, (size_t)n_cols * sizeof(int64_t)));
        BDG_CUDA(cudaMemcpyAsync(st.mu_tmp.ptr, probe_rows, (size_t)n_cols * sizeof(int64_t), cudaMemcpyHostToDevice, sys->stream));
        init_classes<<<(unsigned)ceil_div((int64_t)vec_elems, kThreads), kThreads, 0, sys->stream>>>(
            x0, (int64_t)vec_elems, n, st.panel_width, n_cols, sys->site_class.as<int32_t>(), st.mu_tmp.as<int64_t>());
        BDG_CUDA(cudaStreamSynchronize(sys->stream));  // probe_rows is borrowed only for this call
    } else {
        BDG_CUDA(cudaMemsetAsync(x0, 0, vec_elems * sizeof(double2), sys->stream));
        BDG_TRY(dev_alloc(sys, st.mu_tmp, (size_t)n_cols * sizeof(int64_t)));
        BDG_CUDA(cudaMemcpyAsync(st.mu_tmp.ptr, probe_rows, (size_t)n_cols * sizeof(int64_t), cudaMemcpyHostToDevice, sys->stream));
        init_probes<<<(unsigned)ceil_div(n_cols, 128), 128, 0, sys->stream>>>(x0, n, st.panel_width, n_cols,
                                                                            st.mu_tmp.as<int64_t>());
        BDG_CUDA(cudaStreamSynchronize(sys->stream));  // probe_rows is borrowed only for this call
    }
    BDG_CUDA(cudaGetLastError());
    st.launches += 1;
    // T_1 = H~ T_0 into vec[1] (cur = 1, vec[0] keeps T_0); the even-vector recursion: E_1 = T_2(H~) E_0 and the dot
    // products of steps 0 and 1 (moments 0..3), one step done.
    return advance(sys, true, 0);
}

extern "C" int bdg_cheb_steps(bdg_t *sys, int32_t n_steps, float *elapsed_ms) {
    BDG_ENTER(sys);
    ChebState &st = sys->cheb;
    BDG_REQUIRE(st.active, "bdg_cheb_begin has not been called");
    BDG_REQUIRE(n_steps >= 0, "negative step count");
    BDG_TRY(ensure_dot_capacity(sys, st.steps_done + n_steps + 1));
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    // (the events are destroyed on every path out, failures included)
    struct Events {
        cudaEvent_t &a, &b;
        ~Events() {
            if (a) cudaEventDestroy(a);
            if (b) cudaEventDestroy(b);
        }
    } events{e0, e1};
    if (elapsed_ms) {
        BDG_CUDA(cudaEventCreate(&e0));
        BDG_CUDA(cudaEventCreate(&e1));
        BDG_CUDA(cudaStreamSynchronize(sys->stream));
        BDG_CUDA(cudaEventRecord(e0, sys->stream));
    }
    for (const int target = st.steps_done + n_steps; st.steps_done < target;) BDG_TRY(advance(sys, false, target - st.steps_done));
    if (elapsed_ms) {
        BDG_CUDA(cudaEventRecord(e1, sys->stream));
        BDG_CUDA(cudaEventSynchronize(e1));
        BDG_CUDA(cudaEventElapsedTime(elapsed_ms, e0, e1));
    }
    return BDG_OK;
}

extern "C" int bdg_cheb_reserve(bdg_t *sys, int32_t n_steps) {
    BDG_ENTER(sys);
    BDG_REQUIRE(sys->cheb.active, "bdg_cheb_begin has not been called");
    BDG_REQUIRE(n_steps >= 0, "negative step count");
    return ensure_dot_capacity(sys, sys->cheb.steps_done + n_steps);
}

extern "C" int bdg_cheb_available(bdg_t *sys, int32_t *n_moments) {
    BDG_REQUIRE(sys && n_moments, "null argument");
    *n_moments = sys->cheb.active ? 2 * (sys->cheb.steps_done + 1) : 0;
    return BDG_OK;
}

extern "C" int bdg_cheb_moments_read(bdg_t *sys, int32_t n_moments, int reduce, double *mu, int mu_on_device) {
    BDG_ENTER(sys);
    ChebState &st = sys->cheb;
    BDG_REQUIRE(st.active, "bdg_cheb_begin has not been called");
    BDG_REQUIRE(mu != nullptr, "null output");
    BDG_REQUIRE(n_moments >= 1 && n_moments <= 2 * (st.steps_done + 1), "only %d moments available, %d requested",
                2 * (st.steps_done + 1), n_moments);
    BDG_REQUIRE(reduce == BDG_MU_PER_COLUMN || reduce == BDG_MU_SUM, "unknown reduce mode");
    BDG_TRY(t2_finish_dots(sys));
    const int n_out = reduce ? 1 : st.n_cols;
    const size_t count = (size_t)n_moments * n_out;
    double *dst = mu;
    if (!mu_on_device) {
        BDG_TRY(dev_alloc(sys, st.mu_tmp, count * sizeof(double)));
        dst = st.mu_tmp.as<double>();
    }
    moments_from_dots<<<(unsigned)ceil_div((int64_t)count, kThreads), kThreads, 0, sys->stream>>>(
        st.dots.as<double>(), n_moments, st.n_cols, st.n_panels * st.panel_width, reduce, dst);
    BDG_CUDA(cudaGetLastError());
    st.launches += 1;
    if (!mu_on_device) {
        BDG_CUDA(cudaMemcpyAsync(mu, dst, count * sizeof(double), cudaMemcpyDeviceToHost, sys->stream));
        BDG_CUDA(cudaStreamSynchronize(sys->stream));
    }
    return BDG_OK;
}

extern "C" int bdg_cheb_moments(bdg_t *sys, int kind, int32_t n_cols, const int64_t *probe_rows, uint64_t seed,
                                int64_t col_offset, double scale, int32_t n_moments, int reduce, double *mu,
                                int mu_on_device) {
    BDG_REQUIRE(n_moments >= 1, "need at least one moment");
    BDG_TRY(bdg_cheb_begin(sys, kind, n_cols, probe_rows, seed, col_offset, scale, BDG_KERNEL_AUTO_MOMENTS));
    BDG_TRY(bdg_cheb_steps(sys, std::max(0, (n_moments + 1) / 2 - 1 - sys->cheb.steps_done), nullptr));
    return bdg_cheb_moments_read(sys, n_moments, reduce, mu, mu_on_device);
}

extern "C" int bdg_cheb_vectors(bdg_t *sys, int which, double *out) {
    BDG_ENTER(sys);
    ChebState &st = sys->cheb;
    BDG_REQUIRE(st.active && out, "no active recursion or null output");
    BDG_REQUIRE(which == 0 || which == 1, "which must be 0 (T_n) or 1 (T_{n-1})");
    BDG_REQUIRE(which == 0 || !st.even(), "the even-vector recursion (kernel T2) keeps T_n and T_{n-2}, not T_{n-1}");
    const BsrDev &m = sys->packed;
    const size_t count = (size_t)m.n_sites * 4 * st.n_cols;
    DevBuf tmp;
    BDG_TRY(dev_alloc(sys, tmp, count * sizeof(double2)));
    unpack_vectors<<<(unsigned)ceil_div((int64_t)count, kThreads), kThreads, 0, sys->stream>>>(
        st.vec[which ? st.prev : st.cur].as<double2>(), (int)m.n_sites, st.panel_width, st.n_cols, tmp.as<double2>());
    cudaError_t err = cudaMemcpyAsync(out, tmp.ptr, count * sizeof(double2), cudaMemcpyDeviceToHost, sys->stream);
    if (err == cudaSuccess) err = cudaStreamSynchronize(sys->stream);
    dev_free(sys, tmp);
    BDG_CUDA(err);
    return BDG_OK;
}

extern "C" int bdg_cheb_info(bdg_t *sys, int64_t *n_blocks, int64_t *bytes_per_step, int32_t *panel_width,
                             int32_t *n_panels, int64_t *launches) {
    BDG_ENTER(sys);
    const ChebState &st = sys->cheb;
    BDG_TRY(build_packed(sys));
    const BsrDev &m = sys->packed;
    if (n_blocks) *n_blocks = m.n_blocks;
    if (bytes_per_step)
        *bytes_per_step = 260 * m.n_blocks + 4 * (m.n_sites + 1) + (int64_t)192 * m.n_sites * st.n_cols;
    if (panel_width) *panel_width = st.panel_width;
    if (n_panels) *n_panels = st.n_panels;
    if (launches) *launches = st.launches;
    return BDG_OK;
}

extern "C" int bdg_cheb_format(bdg_t *sys, int32_t *kernel, int64_t *matrix_bytes_per_step, int64_t *n_distinct_blocks) {
    BDG_ENTER(sys);
    const ChebState &st = sys->cheb;
    BDG_REQUIRE(st.active, "bdg_cheb_begin has not been called");
    const BsrDev &m = sys->packed;
    const EllDev &e = sys->ell;
    if (kernel) *kernel = st.even() ? BDG_KERNEL_T2 : st.stepping == Stepping::Pair ? BDG_KERNEL_PAIR : st.kernel;
    if (n_distinct_blocks) *n_distinct_blocks = e.valid ? e.n_unique : 0;
    if (matrix_bytes_per_step) {
        if (st.stepping == Stepping::EvenCube)  // eight 4-byte codes per site, read once per panel and launch (= two steps)
            *matrix_bytes_per_step = e.n_sites * kCubeCodes * 4 * st.n_panels / 2 + e.n_unique * 256;
        else if (st.stepping != Stepping::Single)  // one pass over the codes (and, site-dependent on-site blocks: over those) serves two steps
            *matrix_bytes_per_step = e.n_sites * kPlaneCodes * 4 / 2 + (st.onsite_per_row ? std::min(e.n_unique, e.n_sites) * (st.onsite_diag ? 32 : 256) / 2
                                                                                  : e.n_unique * 256);
        else if (st.kernel == BDG_KERNEL_DICT || st.kernel == BDG_KERNEL_DICT_DIAG)
            *matrix_bytes_per_step = e.n_sites * e.width * 8 + e.n_unique * 256;
        else if (st.kernel == BDG_KERNEL_ELL)
            *matrix_bytes_per_step = e.n_sites * e.width * 260;
        else
            *matrix_bytes_per_step = 260 * m.n_blocks + 4 * (m.n_sites + 1);
    }
    return BDG_OK;
}

extern "C" int bdg_cheb_launched(bdg_t *sys, char *names, int64_t capacity, int64_t *needed) {
    BDG_ENTER(sys);
    const ChebState &st = sys->cheb;
    BDG_REQUIRE(st.active, "bdg_cheb_begin has not been called");
    BDG_REQUIRE(needed != nullptr, "null argument");
    std::string all;
    for (const void *k : st.launched) {
        const char *name = nullptr;
        BDG_CUDA(cudaFuncGetName(&name, k));
        if (!all.empty()) all += '\n';
        all += name;
    }
    *needed = (int64_t)all.size() + 1;
    if (!names) return BDG_OK;
    BDG_REQUIRE(capacity >= *needed, "a buffer of %lld bytes is needed, %lld given", (long long)*needed, (long long)capacity);
    std::memcpy(names, all.c_str(), all.size() + 1);
    return BDG_OK;
}

extern "C" int bdg_cheb_end(bdg_t *sys) {
    BDG_ENTER(sys);
    cheb_release(sys);
    return BDG_OK;
}
