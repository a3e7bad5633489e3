// Chebyshev step on the kernel-native matrix format ("ELL"): fixed-width block rows, diagonal
// block first, blocks stored in MMA B-fragment order.  This is the default step kernel for
// lattice Hamiltonians (every row has <= 8 blocks and almost all rows have the same count);
// ragged / long-row matrices use the generic BSR kernel in cheb.cu.  formats.cu builds the format and
// keeps it current after a scatter.
//
// Formulation.  For block B = Br + i Bi (4x4) and record X = Xr + i Xi (4 components x PW columns)
//     Y^T = X^T B^T :   acc1 = Xr^T * Bop,  acc2 = Xi^T * Bop,   Bop[b][2a]   = Br[a][b]
//                                                               Bop[b][2a+1] = Bi[a][b]
// so that acc1 = (RR[a], IR[a]) and acc2 = (RI[a], II[a]) land in the SAME lane and
//     Re y[a] = acc1.0 - acc2.1,   Im y[a] = acc1.1 + acc2.0
// need no shuffle.  With mma.m8n8k4 (A 8x4 row, B 4x8 col, C 8x8):
//   A fragment: lane l = X[component l%4][column l/4]   = element l of the site record
//   B fragment: lane l = Bop[l%4][l/4]                  = double l of the stored block
//   C fragment: lane l = (column l/4, n = 2(l%4), 2(l%4)+1) -> y[component l%4][column l/4]
// i.e. a lane's output element is the record element it loaded: T_{n+1}[row] is stored, and
// T_{n-1}[row] loaded, with the same fully coalesced 128-bit access, and T_n[row] (needed by the
// dot products) IS the record already fetched for the diagonal block in slot 0.
//
// Per row and panel the warp issues CH 64-bit block loads (one pass over the matrix serves up
// to NP panels: the B fragments stay in registers), CH + 1 128-bit record loads and one 128-bit
// store -- about half the L1 wavefronts of the interleaved-complex formulation in cheb.cu, which
// ncu showed to be the co-limiter next to HBM (l1tex data-pipe wavefronts 77 % at 1.9 GHz).
#include <algorithm>
#include <cstdlib>

#include "bdg_internal.h"
#include "cheb_device.cuh"
#include "cheb_plan.h"

namespace {

__device__ __forceinline__ uint64_t l2_policy(bool evict_first) {
    uint64_t p;
    if (evict_first)
        asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;\n" : "=l"(p));
    else
        asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;\n" : "=l"(p));
    return p;
}

// Matrix blocks: read once per pass, never from L1 again.
__device__ __forceinline__ double ld_block(const double *p, uint64_t policy) {
    double v;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.f64 %0, [%1], %2;\n" : "=d"(v) : "l"(p), "l"(policy));
    return v;
}

// Table blocks (DICT): a few KB..MB re-read by every row that changes its block pattern -- keep in L1/L2.
// L1 prefetch of one 128-byte line (SASS: CCTL.E.PF1) -- no register, no scoreboard slot.
// Predicated for the same reason as ld_table_if below.
__device__ __forceinline__ void prefetch_l1_if(const void *p, unsigned take) {
    asm volatile("{\n .reg .pred p;\n setp.ne.u32 p, %1, 0;\n @p prefetch.global.L1 [%0];\n}\n" ::"l"(p), "r"(take));
}

// Predicated (not branched) so that the row body stays ONE basic block: ptxas schedules per block,
// and a block boundary between the loads and the MMAs lets it issue an MMA -- and stall on its
// operands -- before the last loads of the row have been issued.
__device__ __forceinline__ void ld_table_if(double &v, const double *p, unsigned take) {
    asm volatile("{\n .reg .pred p;\n setp.ne.u32 p, %2, 0;\n @p ld.global.nc.f64 %0, [%1];\n}\n"
                 : "+d"(v)
                 : "l"(p), "r"(take));
}

// DICT = block-dictionary matrix format: `cdata` is the table of DISTINCT blocks (B-fragment order)
// and `ccode[row][slot]` names the table entry of every slot.  The B fragments stay in registers
// from one row of the warp to the next and a slot is re-fetched only when its code changes
// (warp-uniform test), so on a lattice with a few distinct hopping / on-site terms the matrix
// costs 8 bytes per block of HBM traffic instead of 260 and no L1 wavefronts at all.
//
// DIAG (with DICT) = every block outside slot 0 is REAL and DIAGONAL (spin-independent or sigma_3
// hopping without pairing on the bonds: -t sigma_0 becomes diag(-t, -t, t, t)).  Such a block scales
// the lane's own element of the neighbour record, so it costs two DFMA instead of two DMMA (which
// occupy the FP64 pipe 16 cycles each) and the held "fragment" is the lane's diagonal entry from
// `dtab[code][4]`.  Once the dictionary has taken the matrix out of the HBM stream the FP64 pipe is
// the next limiter (ncu: math-pipe-throttle stalls), which this removes for the common models.
//
// SD (with DICT, without DIAG) = every block in slot 0 -- the on-site block -- is real and diagonal (a chemical potential
// and a Zeeman sigma_3 term without on-site pairing: d-wave / p-wave models, Rashba wires) while the hopping blocks are
// general: the on-site product is two multiplications instead of two MMAs (a tenth of the row's FP64-pipe time at five
// blocks per row; the complex-hopping models are the ones the FP64 pipe bounds).  The MMA accumulators START from those
// products, which is what the MMA of a real-diagonal block leaves in them: same sums, same order as DICT.
template <int PW, int CH, int NP, bool DICT, bool DIAG, bool SD = false>
__global__ void __launch_bounds__(kThreads, 4)
cheb_step_ell(const int32_t *__restrict__ cidx, const int32_t *__restrict__ ccode, const double *__restrict__ cdata,
              const double *__restrict__ dtab, const double2 *__restrict__ x_cur, double2 *__restrict__ x_io, int n_sites, int n_panels, double alpha,
              double beta, int first, int stream_matrix, double *__restrict__ partials,
              unsigned *__restrict__ tickets, double *__restrict__ dots_step, const RowWalk wk) {
    constexpr int REC = PW * 4;           // complex elements per site record
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int panel0 = blockIdx.y * NP;
    const size_t plane = (size_t)n_sites * REC;
    const bool x_lane = lane < REC;       // lanes past the record (PW < 8) compute on element 0 and discard
    const int x_elem = x_lane ? lane : 0;
    const uint64_t policy = l2_policy(stream_matrix != 0);
    // Per-row index fetch: lanes 0..CH-1 read the slot's block column, lanes 8..8+CH-1 its code (DICT).
    const int32_t *islot = (DICT && lane >= 8) ? ccode - 8 : cidx;
    const bool ilane = DICT ? ((lane & 7) < CH && lane < 16) : lane < CH;

    // Row traversal (RowWalk, bdg_internal.h): this warp owns one site of the CTA's patch and
    // marches it along x through the item's segment; `row` is the row in hand, `nrow` the one after.
    const int M = wk.Lz * wk.Ly;
    int item = (int)blockIdx.x - (int)gridDim.x, row = -1, row_end = 0;
    auto next_row = [&](int r) -> int {
        if (wk.Lx == 1 && wk.Ly == 1) {  // consecutive rows, one per warp and item
            item += gridDim.x;
            r = item * wk.Pz + warp;
            return item < wk.n_items && r < wk.Lz ? r : -1;
        }
        r += M;
        while (r >= row_end || r < 0) {
            item += gridDim.x;
            if (item >= wk.n_items) return -1;
            const int seg = item / wk.n_patches, p = item - seg * wk.n_patches;
            const int py = p / wk.nPz, pz = p - py * wk.nPz;
            const int z = pz * wk.Pz + warp % wk.Pz, y = py * wk.Py + warp / wk.Pz;
            if (z >= wk.Lz || y >= wk.Ly) continue;  // ragged patch: this warp has no site in it
            const int x0 = seg * wk.seg_len, x1 = min(wk.Lx, x0 + wk.seg_len);
            r = z + y * wk.Lz + x0 * M;
            row_end = z + y * wk.Lz + (x1 - 1) * M + 1;
        }
        return r;
    };
    row = next_row(-1 - M);
    int nrow = row >= 0 ? next_row(row) : -1;
    int jv = 0;
    if (row >= 0 && ilane) jv = __ldg(islot + (size_t)row * CH + lane);

    // March prefetch: the records of a step that are not in L1 yet are the +x neighbour's T_n, the
    // row's own T_{n-1} and -- for the warps on the rim of the patch -- the z / y neighbours owned by
    // other CTAs.  All their addresses are known `wk.prefetch` rows ahead.  Lane groups of LINES lanes
    // (one lane per 128-byte line of a record): 0 = T_n[+M], 1 = T_{n-1}[0], 2 = T_n[z halo], 3 = T_n[y halo].
    constexpr int LINES = (REC * 16 + 127) / 128;
    const int pf_group = lane / LINES;
    int pf_delta = 0;           // row offset of the record this lane prefetches
    bool pf_lane = DICT && NP == 1 && wk.prefetch > 0;  // (the plain kernel streams the matrix: hints only cost it issue slots, measured)
    {
        const int dz = warp % wk.Pz, dy = warp / wk.Pz;
        if (pf_group == 0) pf_delta = M;
        else if (pf_group == 1) pf_lane = pf_lane && !first;
        else if (pf_group == 2) {
            pf_delta = dz == 0 ? -1 : 1;
            pf_lane = pf_lane && wk.Lz > 1 && (dz == 0 || dz == wk.Pz - 1);
        } else if (pf_group == 3) {
            pf_delta = dy == 0 ? -wk.Lz : wk.Lz;
            pf_lane = pf_lane && wk.Ly > 1 && wk.Lx > 1 && (dy == 0 || dy == wk.Py - 1);
        } else {
            pf_lane = false;
        }
    }
    const char *pf_base = reinterpret_cast<const char *>(pf_group == 1 ? x_io : x_cur) + (size_t)(lane % LINES) * 128;

    double d0[NP], d1[NP];
#pragma unroll
    for (int pp = 0; pp < NP; ++pp) d0[pp] = d1[pp] = 0.0;
    double keep[DICT ? CH : 1];  // DICT: B fragments carried from row to row
#pragma unroll
    for (int u = 0; u < (DICT ? CH : 1); ++u) keep[u] = 0.0;
    int jheld = -1;              // DICT: lanes 8.. remember the code of the fragment held for their slot

    for (; row >= 0; row = nrow, nrow = row >= 0 ? next_row(row) : -1) {
        int jn[CH];
#pragma unroll
        for (int u = 0; u < CH; ++u) jn[u] = __shfl_sync(kFull, jv, u);
        double bop[CH];
        if (DICT) {
            // Reload the held fragments only when a code differs from the previous row's (warp-uniform
            // and rare inside a homogeneous region).  The branch sits BEFORE the row's loads so that
            // loads and MMAs still share one basic block.
            const unsigned changed = __ballot_sync(kFull, jv != jheld) >> 8;
            if (changed) {
                jheld = jv;
#pragma unroll
                for (int u = 0; u < CH; ++u) {
                    const int code = __shfl_sync(kFull, jv, 8 + u);
                    const double *entry = ((DIAG && u > 0) || (SD && u == 0)) ? dtab + (size_t)code * 4 + (lane & 3) : cdata + (size_t)code * 32 + lane;
                    ld_table_if(keep[u], entry, changed >> u & 1u);
                }
            }
#pragma unroll
            for (int u = 0; u < CH; ++u) bop[u] = keep[u];
        } else {
            const double *blk = cdata + (size_t)row * CH * 32 + lane;
#pragma unroll
            for (int u = 0; u < CH; ++u) bop[u] = ld_block(blk + u * 32, policy);
        }
        int jnext = 0;
        if (nrow >= 0 && ilane) jnext = __ldg(islot + (size_t)nrow * CH + lane);
        if (DICT && NP == 1) {
            const int prow = row + wk.prefetch + pf_delta;
            prefetch_l1_if(pf_base + ((size_t)panel0 * plane + (size_t)prow * REC) * sizeof(double2),
                           pf_lane && prow >= 0 && prow < n_sites);
            // ... and the index / code lines of the row after next (jnext covers the next one)
            const int irow = row + wk.prefetch + M;
            prefetch_l1_if(islot + (size_t)irow * CH + lane, wk.prefetch > 0 && ilane && irow < n_sites);
        }
        const size_t off = (size_t)row * REC + x_elem;

        // all loads of the NP panels first, then their products
        double2 xv[NP][CH], pv[NP];
        bool on[NP];
#pragma unroll
        for (int pp = 0; pp < NP; ++pp) {
            const int panel = panel0 + pp;
            on[pp] = NP == 1 || panel < n_panels;          // uniform; ragged last group only
            const size_t base = (size_t)(on[pp] ? panel : n_panels - 1) * plane;
#pragma unroll
            for (int u = 0; u < CH; ++u) xv[pp][u] = ld_reuse(x_cur + base + (size_t)jn[u] * REC + x_elem);
            pv[pp] = make_double2(0.0, 0.0);
            if (!first) pv[pp] = ld_plain(x_io + base + off);
        }
#pragma unroll
        for (int pp = 0; pp < NP; ++pp) {
            double a10 = 0.0, a11 = 0.0, a20 = 0.0, a21 = 0.0;
            if (SD) a10 = bop[0] * xv[pp][0].x, a20 = bop[0] * xv[pp][0].y;
#pragma unroll
            for (int u = SD ? 1 : 0; u < (DIAG ? 1 : CH); ++u) {
                dmma_8x8x4(a10, a11, xv[pp][u].x, bop[u]);
                dmma_8x8x4(a20, a21, xv[pp][u].y, bop[u]);
            }
            double yr = a10 - a21, yi = a11 + a20;
            if (DIAG) {
#pragma unroll
                for (int u = 1; u < CH; ++u) {
                    yr = fma(bop[u], xv[pp][u].x, yr);
                    yi = fma(bop[u], xv[pp][u].y, yi);
                }
            }
            if (on[pp] && x_lane) {
                const double2 tn = xv[pp][0];  // slot 0 is the row's own record
                const double2 out = make_double2(alpha * yr - beta * pv[pp].x, alpha * yi - beta * pv[pp].y);
                x_io[(size_t)(panel0 + pp) * plane + off] = out;
                d0[pp] += tn.x * tn.x + tn.y * tn.y;
                d1[pp] += out.x * tn.x + out.y * tn.y;
            }
        }
        jv = jnext;
    }
    // a column's four components sit in one quad of lanes
#pragma unroll
    for (int pp = 0; pp < NP; ++pp) {
        d0[pp] += __shfl_xor_sync(kFull, d0[pp], 1);
        d1[pp] += __shfl_xor_sync(kFull, d1[pp], 1);
        d0[pp] += __shfl_xor_sync(kFull, d0[pp], 2);
        d1[pp] += __shfl_xor_sync(kFull, d1[pp], 2);
    }
#pragma unroll
    for (int pp = 0; pp < NP; ++pp)
        if (NP == 1 || panel0 + pp < n_panels)
            finish_dots<PW>(d0[pp], d1[pp], lane >> 2, x_lane && (lane & 3) == 0, panel0 + pp, n_panels, partials,
                            tickets, dots_step);
}

template <int PW, int NP, bool DICT, bool DIAG, bool SD> EllKernel pick_ch(int width) {
    switch (width) {
        case 3: return cheb_step_ell<PW, 3, NP, DICT, DIAG, SD>;
        case 4: return cheb_step_ell<PW, 4, NP, DICT, DIAG, SD>;
        case 5: return cheb_step_ell<PW, 5, NP, DICT, DIAG, SD>;
        case 6: return cheb_step_ell<PW, 6, NP, DICT, DIAG, SD>;
        case 7: return cheb_step_ell<PW, 7, NP, DICT, DIAG, SD>;
        default: return cheb_step_ell<PW, 8, NP, DICT, DIAG, SD>;
    }
}

template <bool DICT, bool DIAG, bool SD = false> EllKernel pick_shape(int pw, int width) {
    switch (pw) {
        case 1: return pick_ch<1, 1, DICT, DIAG, SD>(width);
        case 2: return pick_ch<2, 1, DICT, DIAG, SD>(width);
        case 4: return pick_ch<4, 1, DICT, DIAG, SD>(width);
        default: return pick_ch<8, 1, DICT, DIAG, SD>(width);
    }
}

// Two panels per pass: the plain format on 8-column panels with rows of >= 6 blocks (ell_configure), so only those widths
// are built.
EllKernel pick_two_panels(int width) {
    switch (width) {
        case 6: return cheb_step_ell<8, 6, 2, false, false, false>;
        case 7: return cheb_step_ell<8, 7, 2, false, false, false>;
        default: return cheb_step_ell<8, 8, 2, false, false, false>;
    }
}

// fmt: BDG_KERNEL_ELL, BDG_KERNEL_DICT or BDG_KERNEL_DICT_DIAG; np: panels per pass (ell_configure); self_diag: DICT with
// real-diagonal on-site blocks (SD)
EllKernel pick_ell(int fmt, int pw, int np, int width, bool self_diag) {
    if (fmt == BDG_KERNEL_DICT_DIAG) return pick_shape<true, true>(pw, width);
    if (fmt == BDG_KERNEL_DICT) return self_diag ? pick_shape<true, false, true>(pw, width) : pick_shape<true, false>(pw, width);
    return np == 2 ? pick_two_panels(width) : pick_shape<false, false>(pw, width);
}

// Plan the row traversal for `slots` resident CTAs per panel group (RowWalk, bdg_internal.h).
RowWalk plan_walk(const bdg_system *sys, int n_sites, int64_t slots, const PlanSwitches &sw) {
    RowWalk w;
    const int Lx = sys->cubic[0], Ly = sys->cubic[1], Lz = sys->cubic[2];
    const bool cubic = (int64_t)Lx * Ly * Lz == n_sites && n_sites > 0;
    if (!cubic || Ly * Lz < 2 * kWarps || Lx < 8 || !sw.ell_walk) {
        // consecutive rows, one per warp: the wavefront sweep of cheb.cu
        w.Lz = std::max(n_sites, 1);
        w.Pz = kWarps;
        w.nPz = (int)ceil_div(w.Lz, kWarps);
        w.n_patches = w.n_items = w.nPz;
        return w;
    }
    w.Lx = Lx, w.Ly = Ly, w.Lz = Lz;
    w.Pz = sw.ell_pz > 0 ? std::min(sw.ell_pz, kWarps) : Lz == 1 ? 1 : (Ly == 1 ? kWarps : 2);
    while (kWarps % w.Pz) --w.Pz;
    w.Py = kWarps / w.Pz;
    w.nPz = (int)ceil_div(Lz, w.Pz);
    w.n_patches = w.nPz * (int)ceil_div(Ly, w.Py);
    // Segment length: long segments amortise the two cold columns at the start of an item, many
    // items balance the CTAs.  Score = (share of CTA slots doing useful work) x (1 - cold share).
    double best = -1.0;
    const int forced = sw.ell_seg;
    for (int n_seg = 1; n_seg <= std::max(1, Lx / 8); ++n_seg) {
        const int len = forced > 0 ? forced : (int)ceil_div(Lx, n_seg);
        const int64_t items = (int64_t)w.n_patches * ceil_div(Lx, len);
        const double balance = (double)items / (double)(ceil_div(items, slots) * slots);
        const double score = balance * len / (len + 2.0);
        if (score > best) {
            best = score;
            w.seg_len = len;
            w.n_items = (int)items;
        }
        if (forced > 0) break;
    }
    w.prefetch = std::max(0, sw.ell_prefetch) * Ly * Lz;
    return w;
}

}  // namespace

// The single-step kernel of the current recursion, its panels per group, grid and row traversal.
int ell_configure(bdg_system *sys, const PlanSwitches &sw) {
    ChebState &st = sys->cheb;
    const EllDev &e = sys->ell;
    // One panel per pass, each panel group marching the lattice on its own CTAs: with the marching
    // traversal and the L1 prefetch this beats sharing the block registers between panels for every
    // dictionary workload measured (profiles/r01/quickperf_np_v2.log).  The plain kernel on 3-D
    // lattices (long rows: more block bytes per record byte) still gains from two panels per pass.
    const bool dict = st.kernel != BDG_KERNEL_ELL;
    const int panels_per_group = !dict && st.panel_width == 8 && st.n_panels >= 2 && e.width >= 6 ? 2 : 1;  // (pick_two_panels)
    const int n_groups = (int)ceil_div(st.n_panels, panels_per_group);
    const EllKernel k = pick_ell(st.kernel, st.panel_width, panels_per_group, e.width, e.self_diag_usable && sw.ell_sd);
    int per_sm = 1;
    BDG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, kThreads, 0));
    per_sm = std::max(per_sm, 1);
    const int64_t slots = std::max<int64_t>(1, (int64_t)sys->sm_count * per_sm / n_groups);
    st.walk = plan_walk(sys, (int)e.n_sites, slots, sw);
    const int gx = (int)std::min<int64_t>(slots, st.walk.n_items);
    st.ell_step = {k, dim3((unsigned)gx, (unsigned)n_groups), kThreads, 0};
    st.partial_runs = std::max(st.partial_runs, gx);
    return BDG_OK;
}

int ell_launch_step(bdg_system *sys, bool first, const void *x_cur, void *x_io, double *dots_step) {
    ChebState &st = sys->cheb;
    const EllDev &e = sys->ell;
    const bool dict = st.kernel != BDG_KERNEL_ELL;
    const Launch<EllKernel> &l = st.ell_step;
    note_launch(st, reinterpret_cast<const void *>(l.fn));
    // Stream the matrix through L2 (evict-first) only when nothing will read it again soon: one
    // group per pass and a matrix that cannot stay resident in the 126 MB L2 anyway.
    const size_t matrix_bytes = (size_t)e.n_sites * e.width * 260;
    const int stream_matrix = l.grid.y == 1 && matrix_bytes > (size_t)64 << 20;
    l.fn<<<l.grid, l.threads, l.smem, sys->stream>>>(e.idx.as<int32_t>(), dict ? e.code.as<int32_t>() : nullptr,
                                                     dict ? e.table.as<double>() : e.data.as<double>(), e.dtab.as<double>(),
                                                     static_cast<const double2 *>(x_cur), static_cast<double2 *>(x_io),
                                                     (int)e.n_sites, st.n_panels, (first ? 1.0 : 2.0) / st.scale, first ? 0.0 : 1.0,
                                                     first ? 1 : 0, stream_matrix, st.partials.as<double>(),
                                                     st.tickets.as<unsigned>(), dots_step, st.walk);
    BDG_CUDA(cudaGetLastError());
    return BDG_OK;
}
