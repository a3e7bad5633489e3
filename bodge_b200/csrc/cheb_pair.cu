// Two Chebyshev steps per pass over the vectors ("pair step", SURVEY 8f-4: temporal blocking).
//
//     T_{n+1} = 2 H~ T_n - T_{n-1},     T_{n+2} = 2 H~ T_{n+1} - T_n
//
// in ONE launch, on the block-dictionary matrix format of cheb_ell.cu.  A single-step kernel moves
// three vector passes per step (read T_n, read T_{n-1}, write T_{n+1}); this one moves four per TWO
// steps (read T_{n-1}, T_n; write T_{n+1}, T_{n+2}) because T_{n+1} never has to come back from HBM:
// it is consumed out of shared memory.  With the matrix already out of the HBM stream (dictionary
// format) that is the only way past the one-pass roofline of the step.
//
// Geometry.  Lattices whose x-planes are one-dimensional (Lz = 1 or Ly = 1; M >= 3 sites per plane, Lx >= 3 planes),
// treated as a TORUS: open and periodic stencils run the same code, the matrix (direction codes) decides what is
// connected.  The plane is cut into patches of P owned sites; a CTA marches one patch along a segment of x:
//
//   iteration i:  [A] T_{n+1} of plane x0 - 1 + i for the P owned sites AND one halo site on either side, from three
//                     T_n planes (P + 4 sites each) staged in a shared-memory ring of 8 planes by bulk async copies
//                     (TMA: cp.async.bulk, one contiguous 9 KB run per plane -- plus one small run from the opposite
//                     side of the plane for the first / last patch --, seven planes ahead, completion on an mbarrier),
//                     and T_{n-1} of the warp's rows, which only this warp reads: straight to registers, one plane
//                     ahead; the result goes to a shared-memory ring (4 planes) and, for owned sites of owned planes,
//                     to HBM;
//                 __syncthreads; the plane [A] no longer needs is replaced by the plane eight ahead
//                 [B] T_{n+2} of the plane one behind, for the owned sites, from the T_{n+1} ring's three planes -- of which
//                     only the middle one, written an iteration ago, is read at other warps' sites -- and the T_n records
//                     [A] read as its x-1 neighbours (kept in registers across the barrier).
//
// The halo T_{n+1} values (one site either side in y, one plane either side of the segment in x)
// are recomputed, not exchanged: (P+2)/P x (len+2)/len redundant work on sub-step [A], no
// inter-CTA dependency, deterministic.  Because a neighbouring CTA may still need T_{n-1} / T_n of
// a site after its owner has produced T_{n+1} / T_{n+2} there, the outputs go to two further
// buffers (four vector buffers in rotation) instead of in place.
//
// Arithmetic per row is exactly that of cheb_step_ell<.., DICT, DIAG> (same fragments, same order,
// same update expression): on open lattices the vectors are bit-identical to the single-step dictionary kernels'
// (where a neighbour wraps around, the terms of a row are added in stencil direction here and in ascending block
// column there: equal to rounding); the dot products are summed over a different partition of the rows (agree to
// rounding).
//
// The other shapes, hand-overs between [A] and [B] and prefetch distances that were measured against this one, and
// why none was kept, are in DESIGN 4.1-iv.
#include <algorithm>
#include <array>
#include <cstdlib>
#include <type_traits>
#include <vector>

#include "bdg_internal.h"
#include "cheb_device.cuh"
#include "cheb_plan.h"
#include "cheb_smem.cuh"
#include "work_lists.h"

namespace {

constexpr int kRecBytes = 512;  // one site record at PW = 8: 8 columns x 4 components x complex128
constexpr int kRing = 4;        // planes of the T_{n+1} ring (three read by [B], one being written)
constexpr int kRingN = 8;       // planes of the T_n ring: three in use, five in flight (power of two)
// 8 warps x 2 sites per CTA, two CTAs per SM: one computes while the other waits at its barrier.  The shape sweep
// (profiles/r01/s4_pair_shape_sweep.log: 16 x 2 one CTA per SM -2 %, 8 x 3 -11 %, 12 x 1 with 24 warps per SM -14 %,
// 6 x 2 with three CTAs per SM -15 %) and the 12-warp shape with its own records in registers (0.159 against 0.141
// ms/step, DESIGN 4.1-iv) left this one ahead.
constexpr int kPairWarps = 8, kPairSites = 2, kPairMinBlocks = 2;

// B fragments of the S rows a warp handles (cheb_ell.cu: DICT / DIAG), held in registers from plane to
// plane and reloaded only when a code differs from the held one.  Lane s * 5 + u carries the code of
// row s, direction u; code < 0 = no block.  SELF: the on-site fragments (u = 0) are not held -- they are
// fetched per row, one plane ahead (self_fragments) -- so their codes do not take part in the test.
template <bool DIAG, bool SELF, int S, bool SD = false>
__device__ __forceinline__ void hold_fragments(int jv, int &jheld, double (&keep)[S][kPlaneCodes], const double *__restrict__ table,
                                               const double *__restrict__ dtab, int lane, bool self_lane) {
    const unsigned changed = __ballot_sync(kFull, jv != jheld && !(SELF && self_lane));
    if (changed) {
        jheld = jv;
#pragma unroll
        for (int s = 0; s < S; ++s) {
#pragma unroll
            for (int u = SELF ? 1 : 0; u < kPlaneCodes; ++u) {
                const int code = __shfl_sync(kFull, jv, s * kPlaneCodes + u);
                const unsigned take = changed >> (s * kPlaneCodes + u) & 1u;
                const size_t c = (size_t)max(code, 0);
                const double *entry = ((DIAG && u > 0) || (SD && u == 0)) ? dtab + c * 4 + (lane & 3) : table + c * 32 + lane;
                ld_table_pred(keep[s][u], entry, take && code >= 0);
                if (take && code < 0) keep[s][u] = 0.0;
            }
        }
    }
}

// SELF: this lane's double of the on-site B fragment of row s, straight from the table by the row's code
// (-1: no diagonal block -> 0).  Issued a plane ahead of its use; with every on-site block distinct (disorder,
// self-consistent gap) this is the 256-byte-per-site stream the matrix cannot do without, with a phase winding
// or a layered structure it hits in L1 / L2.
template <int S, bool SD = false>
__device__ __forceinline__ void self_fragments(int jv, double (&f)[S], const double *__restrict__ table, const double *__restrict__ dtab,
                                               int lane) {
#pragma unroll
    for (int s = 0; s < S; ++s) {
        const int code = __shfl_sync(kFull, jv, s * kPlaneCodes);
        f[s] = 0.0;
        ld_table_pred(f[s], SD ? dtab + (size_t)max(code, 0) * 4 + (lane & 3) : table + (size_t)max(code, 0) * 32 + lane, code >= 0);
    }
}

// y = sum_u B_u x_u for this lane's element; order and operations of cheb_step_ell (directions: self, x-1, y-1,
// y+1, x+1 = ascending block column on an open lattice), in stages so that sub-step [A] can wait for its newest plane
// only before the last term: begin (self), add x 4, end.
// SD (without DIAG): the on-site block is real and diagonal (cheb_ell.cu: SD) -- its product is two multiplications, and
// the accumulators of the hopping blocks' MMAs start from them (what the MMA of such a block leaves there).
template <bool DIAG, bool SD = false> struct RowSum {
    double a10 = 0.0, a11 = 0.0, a20 = 0.0, a21 = 0.0, yr = 0.0, yi = 0.0;
    __device__ __forceinline__ void begin(const double2 &x0, double b0) {
        if (SD && !DIAG) {
            a10 = b0 * x0.x, a20 = b0 * x0.y;
            return;
        }
        dmma_8x8x4(a10, a11, x0.x, b0);
        dmma_8x8x4(a20, a21, x0.y, b0);
        if (DIAG) yr = a10 - a21, yi = a11 + a20;
    }
    __device__ __forceinline__ void add(const double2 &x, double b) {
        if (DIAG) {
            yr = fma(b, x.x, yr);
            yi = fma(b, x.y, yi);
        } else {
            dmma_8x8x4(a10, a11, x.x, b);
            dmma_8x8x4(a20, a21, x.y, b);
        }
    }
    __device__ __forceinline__ void end() {
        if (!DIAG) yr = a10 - a21, yi = a11 + a20;
    }
};

template <bool DIAG, bool SD = false>
__device__ __forceinline__ void row_product(const double2 &x0, const double2 &x1, const double2 &x2, const double2 &x3,
                                            const double2 &x4, double b0, const double (&bop)[kPlaneCodes], double &yr, double &yi) {
    RowSum<DIAG, SD> r;
    r.begin(x0, b0);
    r.add(x1, bop[1]);
    r.add(x2, bop[2]);
    r.add(x3, bop[3]);
    r.add(x4, bop[4]);
    r.end();
    yr = r.yr;
    yi = r.yi;
}

// NW warps per CTA, S = 2 ADJACENT sites per warp and plane: W = 2 NW sites per plane in sub-step [A]
// (P <= W - 2 of them owned).  Dynamic shared memory: kRingN planes of W + 2 records (T_n), kRing
// planes of W records (T_{n+1}), two guard records, one mbarrier per T_n plane and one more: 105 KB, so two
// CTAs share an SM.
//
// Geometry is a TORUS: planes x and in-plane sites y are taken modulo Lx and M, so the halo of the first /
// last patch and of the first / last segment is the opposite face of the lattice (staged by its own small bulk
// copy).  What is connected is decided by the matrix alone: it arrives as `dcode[row][kPlaneCodes]`, the dictionary
// code of the row's block in each stencil direction (self, x-1, y-1, y+1, x+1; kNoBlock = none), so the reference's
// periodic skeleton with the edges filled in (bodge/lattice.py:161-197) and the open lattice it leaves when they
// are not run the same code: a direction without a block meets a zero fragment (whatever finite vector value
// sits at the wrapped position is multiplied by zero; the rings are cleared once).  The records a row needs sit
// at fixed offsets from its own in the rings -- no per-row index arithmetic -- and the two sites of a warp
// share their in-plane neighbours (4 loads for 6 operands).  Warps whose site does not exist (ragged last patch)
// compute on whatever the rings hold and store nothing: the row body has no branches.
//
// An item = (patch, segment [x0, x0 + len)).  Iteration i = 0 .. len + 1 of an item:
//   [A] plane x0 - 1 + i from the T_n planes t = i, i + 1, i + 2 of the item (t <-> plane x0 - 2 + t);
//       stored / counted in the dot products for 1 <= i <= len
//   [B] plane x0 - 2 + i (i >= 2) from the T_{n+1} planes of iterations i - 2, i - 1, i
// T_n planes occupy ring slots in the order they are consumed, across items (`cnt`): slot = count & 7, mbarrier
// parity = (count >> 3) & 1.
//
// MODE 1 ("T2", the doubled-argument recursion) runs the same two sub-steps on the EVEN vectors only:
//     E_j = T_2j(H~) x,   E_{j+1} = 2 T_2(H~) E_j - E_{j-1} = 4 H~ (H~ E_j) - 2 E_j - E_{j-1}
// [A] u = H~ E_j (halo included, shared memory only, never stored), [B] E_{j+1} for the owned rows, written in
// place over E_{j-1} (read by its owner alone).  One launch is still two applications of H~ and four dot products
//     a = <E_j, E_j>, c = <u, E_j>, b = <E_{j+1}, E_j>, d = <E_{j+1}, u>
// from which the same four moments follow (cheb.cu: t2_normalize), but it moves THREE vector passes instead
// of four, and two vector buffers suffice.  `first`: E_1 = T_2(H~) E_0 = 2 H~ u - E_0 (E_{-1} = E_1).
//
// LISTED: the CTA's pieces come from the work lists of PairWalk (balanced plan, grid = (n_ctas, 1)); otherwise they are
// computed from the item index (classic plan, grid = (CTAs per panel, panels)) -- kept as arithmetic on kernel parameters
// because values loaded from memory leave the uniform datapath and the plane loop's predicates with them (+2 % time).
template <bool DIAG, bool SELF, int MODE, bool SD = false, bool LISTED = false>
__global__ void __launch_bounds__(kPairWarps * 32, kPairMinBlocks)
cheb_pair_step(const int32_t *__restrict__ dcode, const double *__restrict__ table, const double *__restrict__ dtab,
               const double2 *__restrict__ xa /* T_{n-1} */, const double2 *__restrict__ xb /* T_n */,
               double2 *__restrict__ xc /* T_{n+1} */, double2 *__restrict__ xd /* T_{n+2} */, int n_sites, int n_panels,
               double alpha, double alpha2, double csub, int first, double *__restrict__ partials, unsigned *__restrict__ tickets,
               double *__restrict__ dots_step, const PairWalk wk) {
    // MODE 1: E_{j+1} = alpha2 H~u - (csub E_j + E_{j-1}); csub = 2, or 1 in the first launch, where E_{-1} is never loaded (= 0)
    constexpr int NW = kPairWarps, S = kPairSites, W = NW * S, R = kRecBytes;
    constexpr uint32_t PLANE_N = (W + 2) * R, PLANE_W = W * R;
    extern __shared__ __align__(128) unsigned char pair_smem[];
    const uint32_t sTn = smem_u32(pair_smem);         // T_n planes, local site l2 = y - (y0 - 2)
    const uint32_t sT1 = sTn + kRingN * PLANE_N + R;  // guard record, then T_{n+1} planes (computed here), local site l = y - (y0 - 1)
    const uint32_t sBar = sT1 + kRing * PLANE_W + R;  // guard record (halo rows of [B] read one before / past the ring), then one mbarrier per T_n slot

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // LISTED: the panel of the pieces in hand and the run (= partial-sum slot) they belong to
    int panel = -1, run = -1;

    for (uint32_t o = threadIdx.x * 16u; o < kRingN * PLANE_N + kRing * PLANE_W + 2 * R; o += NW * 32 * 16u)
        sts_rec(sTn + o, make_double2(0.0, 0.0));
    if (threadIdx.x == 0) {
#pragma unroll
        for (int r = 0; r < kRingN; ++r) mbar_init(sBar + 8 * r, 1);
        // Nothing waits on this ninth barrier; it is initialised so that the kernel's code stays the code DESIGN 4.1-iv measured.
        mbar_init(sBar + 8 * kRingN, NW * 32);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");  // the clears are ordered before the bulk copies
    __syncthreads();
    uint32_t cnt = 0;  // T_n planes consumed by the items before this one
    const size_t gstep = (size_t)wk.M * 32;
    double d0 = 0.0, d1 = 0.0, d2 = 0.0, d3 = 0.0;

    const int l0 = S * warp;  // this warp's sites: l0, l0 + 1
    // own-record addresses of site l0 in slot 0 of each ring (+ lane's 16 bytes)
    uint32_t aN = sTn + (uint32_t)(l0 + 1) * R + (uint32_t)lane * 16u;
    uint32_t a1 = sT1 + (uint32_t)l0 * R + (uint32_t)lane * 16u;
    pin(aN), pin(a1);

    double keep[S][kPlaneCodes];
    int jheld = -2;
#pragma unroll
    for (int s = 0; s < S; ++s)
#pragma unroll
        for (int u = 0; u < kPlaneCodes; ++u) keep[s][u] = 0.0;
    // lanes 0 .. 5 S - 1 carry the codes of the warp's rows: lane = s * 5 + direction
    const int csite = lane / kPlaneCodes, cdir = lane - csite * kPlaneCodes;
    const bool code_lane = lane < S * kPlaneCodes, self_lane = cdir == 0;
    const int plane_codes = wk.M * kPlaneCodes, all_codes = wk.Lx * plane_codes;

    const int item0 = LISTED ? wk.lists.cta_begin[blockIdx.x] : (int)blockIdx.x, item1 = LISTED ? wk.lists.cta_begin[blockIdx.x + 1] : wk.n_items;
    for (int item = item0; item < item1; item += LISTED ? 1 : (int)gridDim.x) {
        int4 piece;  // panel, patch, x0, len
        if (LISTED) {
            piece = wk.lists.pieces[item];  // (run, patch, x0, len)
            if (piece.x != run) {
                if (run >= 0) {
                    flush_dots<NW, 8>(d0, d1, d2, d3, pair_smem, run, wk.lists.panel_runs[panel], wk.lists.panel_runs[panel + 1], panel, n_panels, partials,
                                      tickets, dots_step);
                    d0 = d1 = d2 = d3 = 0.0;
                }
                run = piece.x;
                panel = wk.lists.run_panel[run];
            }
            piece.x = panel;
        } else {
            const int seg = item / wk.n_patches;
            piece.x = (int)blockIdx.y, piece.y = item - seg * wk.n_patches, piece.z = seg * wk.seg_len;
            piece.w = min(wk.Lx, piece.z + wk.seg_len) - piece.z;
        }
        const size_t pbase = (size_t)piece.x * n_sites * 32;
        const double2 *const ta = xa + pbase, *const tb = xb + pbase;
        double2 *const tc = xc + pbase, *const td = xd + pbase;  // MODE 1: td = ta (E_{j+1} over E_{j-1}), tc unused
        const int patch = piece.y;
        // Local site l = 1 of a patch is y0.  On a plane with OPEN ends (wk.open: no block wraps around in-plane) the site
        // below the first patch / above the last one does not exist, so those two patches own their rim site too (l = 0 resp.
        // l = P + 1) instead of recomputing a halo value nobody needs: n P + 2 sites in n patches (100 sites: 7 instead of 8).
        const int y0 = patch * wk.P + wk.open, x0 = piece.z, len = piece.w;
        const int own_lo = wk.open && patch == 0 ? 0 : 1, own_hi = wk.P + (wk.open && patch == wk.n_patches - 1 ? 1 : 0);
        const int n_planes = len + 4;  // T_n planes x0 - 2 .. x0 + len + 1 (mod Lx); plane t -> ring slot (cnt + t) % kRingN
        // In-plane run of a T_n plane: y = y0 - 2 .. ye + 1 (ye = end of the owned sites; at most the W + 2 records of a ring
        // plane), l2 = y - (y0 - 2); the part below 0 / from M on comes from the opposite side of the plane (its own small
        // bulk copy).
        const int ye = min(wk.M, y0 + own_hi), span = min(ye - y0 + 4, W + 2);
        const int n_lo = max(0, 2 - y0), n_hi = max(0, y0 - 2 + span - wk.M);
        const double2 *src_lo = tb + (ptrdiff_t)(y0 - 2 + wk.M) * 32, *src_main = tb + (ptrdiff_t)(y0 - 2 + n_lo) * 32,
                      *src_hi = tb + (ptrdiff_t)(y0 - 2 + span - n_hi - wk.M) * 32;
        // One elected thread stages a plane: expect the bytes on the slot's barrier, then up to three bulk copies.
        auto issue = [&](int t) {
            if (warp == 0 && t < n_planes) {
                int xw = x0 - 2 + t;
                xw += xw < 0 ? wk.Lx : 0;
                xw -= xw >= wk.Lx ? wk.Lx : 0;
                const size_t po = (size_t)xw * gstep;
                const uint32_t r = (cnt + (uint32_t)t) & (kRingN - 1);
                const uint32_t dst = sTn + r * PLANE_N, bar = sBar + 8 * r;
                if (lane == 0) {
                    mbar_expect_tx(bar, (uint32_t)span * R);
                    bulk_g2s(dst + (uint32_t)n_lo * R, src_main + po, (uint32_t)(span - n_lo - n_hi) * R, bar);
                    if (n_lo) bulk_g2s(dst, src_lo + po, (uint32_t)n_lo * R, bar);
                    if (n_hi) bulk_g2s(dst + (uint32_t)(span - n_hi) * R, src_hi + po, (uint32_t)n_hi * R, bar);
                }
            }
        };
        auto wait = [&](int t) {
            if (t < n_planes) {
                const uint32_t c = cnt + (uint32_t)t;
                mbar_wait(sBar + 8 * (c & (kRingN - 1)), (c >> 3) & 1u);
            }
        };

        __syncthreads();  // every warp is done with the previous item's planes
        for (int t = 0; t < kRingN; ++t) issue(t);

        // Site l0 + s of this warp: y = y0 - 1 + l0 + s (mod M).  Owned = inside the patch and the lattice.
        const int ya = y0 - 1 + l0;
        bool owned[S];
#pragma unroll
        for (int s = 0; s < S; ++s) owned[s] = l0 + s >= own_lo && l0 + s <= own_hi && ya + s < wk.M;
        // code index of this lane's (row, direction) in plane 0; rows past the halo (ragged patch) wrap anywhere valid
        int yl = (ya + csite) % wk.M;
        yl += yl < 0 ? wk.M : 0;
        const int coff = yl * kPlaneCodes + cdir;
        int cplane = x0 - 1;  // plane of [A] in iteration 0
        cplane += cplane < 0 ? wk.Lx : 0;
        cplane *= plane_codes;
        // codes of the planes of [A] in this iteration, [B] (one plane behind), and of the next two planes of [A]: loaded
        // two planes ahead, so that the on-site fragment fetch of the next plane (SELF) never waits for its code
        int jvA = -1, jvB = -1, jnext = -1;
        if (code_lane) jvA = __ldg(dcode + cplane + coff);
        cplane += plane_codes;
        cplane -= cplane >= all_codes ? all_codes : 0;
        if (code_lane) jnext = __ldg(dcode + cplane + coff);
        double fsA[S], fsB[S], fsN[S];  // SELF: on-site fragments of the planes of [A], [B] and of the next [A]
#pragma unroll
        for (int s = 0; s < S; ++s) fsA[s] = fsB[s] = fsN[s] = 0.0;
        if (SELF) self_fragments<S, SD>(jvA, fsA, table, dtab, lane);
        // Global element of (plane x0 - 1, site ya): T_{n+1} / E_{j-1} / E_{j+1} of the warp's rows; only owned rows of
        // owned planes are dereferenced through it.  The second row sits 32 elements on.
        const ptrdiff_t gbase = ((ptrdiff_t)(x0 - 1) * wk.M + ya) * 32 + lane;
        const double2 *pin_ = ta + gbase;                       // MODE 1: E_{j-1}(plane of [A])
        double2 *pout1 = tc + gbase;                            // MODE 0: T_{n+1}(plane of [A])
        double2 *pout2 = td + gbase - (ptrdiff_t)gstep;         // T_{n+2} / E_{j+1}(plane of [B]) = one plane behind [A]
        // MODE 0: T_{n-1} of ALL rows [A] computes (halo rows and halo planes included), wrapped like the codes;
        // MODE 1: E_{j-1} of the owned rows of the plane [B] works on.  Both one plane ahead (pvn).
        int yw[S];
#pragma unroll
        for (int s = 0; s < S; ++s) {
            yw[s] = (ya + s) % wk.M;
            yw[s] += yw[s] < 0 ? wk.M : 0;
        }
        int xprev = x0 - 1;  // wrapped plane of [A]
        xprev += xprev < 0 ? wk.Lx : 0;
        double2 pv[S], pvn[S];  // MODE 1: E_{j-1} of the plane of [B] in this / in the next iteration
#pragma unroll
        for (int s = 0; s < S; ++s) {
            pv[s] = pvn[s] = make_double2(0.0, 0.0);
            if (MODE == 0) pvn[s] = ld_prev(ta + ((size_t)xprev * wk.M + yw[s]) * 32 + lane);
        }
        wait(0);
        wait(1);

        for (int i = 0; i <= len + 1; ++i, pin_ += gstep, pout1 += gstep, pout2 += gstep) {
            const bool store = i >= 1 && i <= len;
            if (MODE == 1) {
                // E_{j-1} of the plane of [A]: [B] of the NEXT iteration works on that plane (and overwrites it) -- issued
                // here, an iteration and a half ahead of its use (half an iteration does not cover the HBM latency: measured)
#pragma unroll
                for (int s = 0; s < S; ++s) {
                    pv[s] = pvn[s];
                    if (store && owned[s] && !first) pvn[s] = ld_prev_rw(pin_ + 32 * s);
                }
            } else {  // T_{n-1} of the next plane of [A], one iteration ahead
                if (i <= len) {
                    xprev += 1;
                    xprev -= xprev >= wk.Lx ? wk.Lx : 0;
                }
#pragma unroll
                for (int s = 0; s < S; ++s) {
                    pv[s] = pvn[s];
                    if (i <= len) pvn[s] = ld_prev(ta + ((size_t)xprev * wk.M + yw[s]) * 32 + lane);
                }
            }
            int jn2 = -1;
            cplane += plane_codes;
            cplane -= cplane >= all_codes ? all_codes : 0;
            if (code_lane && i < len) jn2 = __ldg(dcode + cplane + coff);
            if (SELF) self_fragments<S, SD>(jnext, fsN, table, dtab, lane);
            double2 tn[S] = {};  // T_n of the warp's rows in the plane of [B] = the records [A] reads as its x-1 neighbours
            double2 out[S] = {};  // T_{n+1} of the warp's rows in the plane of [A]
            // [B]: update, store and dot products of row s from its product (yr, yi) and its own T_{n+1} record
            auto finish_b = [&](int s, double yr, double yi, const double2 &own1) {
                const double2 t = tn[s];
                double2 out;
                if (MODE == 0) {
                    out = make_double2(fma(alpha, yr, -t.x), fma(alpha, yi, -t.y));
                } else {
                    const double2 sub = make_double2(fma(csub, t.x, pv[s].x), fma(csub, t.y, pv[s].y));
                    out = make_double2(fma(alpha2, yr, -sub.x), fma(alpha2, yi, -sub.y));
                }
                if (owned[s]) {
                    pout2[32 * s] = out;
                    if (MODE == 0) {
                        d2 = fma(own1.x, own1.x, fma(own1.y, own1.y, d2));
                    } else {
                        d2 = fma(out.x, t.x, fma(out.y, t.y, d2));
                    }
                    d3 = fma(out.x, own1.x, fma(out.y, own1.y, d3));
                }
            };
            {
                const uint32_t c = cnt + (uint32_t)i;
                const uint32_t nm = aN + (c & (kRingN - 1)) * PLANE_N;
                const uint32_t n0 = aN + ((c + 1) & (kRingN - 1)) * PLANE_N;
                const uint32_t np = aN + ((c + 2) & (kRingN - 1)) * PLANE_N;
                hold_fragments<DIAG, SELF, S, SD>(jvA, jheld, keep, table, dtab, lane, self_lane);
                double2 c_[S + 2], q[S];  // c_[1 + s] = the own record of site s; c_[0], c_[S + 1] = the warp's in-plane neighbours
#pragma unroll
                for (int k = 0; k < S + 2; ++k) c_[k] = lds_rec(n0 + (uint32_t)(k - 1) * R);
#pragma unroll
                for (int s = 0; s < S; ++s) tn[s] = lds_rec(nm + (uint32_t)s * R);
                const uint32_t t1 = a1 + (uint32_t)(i & (kRing - 1)) * PLANE_W;
                // The newest plane (x+1 neighbours) feeds the LAST term of a row: its barrier is waited for only after the
                // other four terms are under way (+1 %: profiles/r02/21_latewait.log).
                RowSum<DIAG, SD> rs[S];
#pragma unroll
                for (int s = 0; s < S; ++s) {
                    rs[s].begin(c_[1 + s], SELF ? fsA[s] : keep[s][0]);
                    rs[s].add(tn[s], keep[s][1]);
                    rs[s].add(c_[s], keep[s][2]);
                    rs[s].add(c_[2 + s], keep[s][3]);
                }
                wait(i + 2);
#pragma unroll
                for (int s = 0; s < S; ++s) q[s] = lds_rec(np + (uint32_t)s * R);
#pragma unroll
                for (int s = 0; s < S; ++s) {
                    double yr, yi;
                    rs[s].add(q[s], keep[s][4]);
                    rs[s].end();
                    yr = rs[s].yr, yi = rs[s].yi;
                    if (MODE == 0) out[s] = make_double2(fma(alpha, yr, -pv[s].x), fma(alpha, yi, -pv[s].y));
                    else out[s] = make_double2(alpha * yr, alpha * yi);
                    sts_rec(t1 + (uint32_t)s * R, out[s]);
                }
                if (store) {
#pragma unroll
                    for (int s = 0; s < S; ++s) {
                        if (owned[s]) {
                            if (MODE == 0) pout1[32 * s] = out[s];
                            d0 = fma(c_[1 + s].x, c_[1 + s].x, fma(c_[1 + s].y, c_[1 + s].y, d0));
                            d1 = fma(out[s].x, c_[1 + s].x, fma(out[s].y, c_[1 + s].y, d1));
                        }
                    }
                }
            }
            __syncthreads();  // T_{n+1} of this plane complete in the ring
            // ... and [A] is done in every warp: plane i (its x-1 neighbours) is dead, its slot takes plane i + 8 -- seven
            // planes in flight beyond the one in use.
            issue(i + kRingN);
            if (i >= 2) {
                const uint32_t t0 = a1 + (uint32_t)((i - 1) & (kRing - 1)) * PLANE_W;
                const uint32_t tm = a1 + (uint32_t)((i - 2) & (kRing - 1)) * PLANE_W;
                const uint32_t tp = a1 + (uint32_t)(i & (kRing - 1)) * PLANE_W;
                hold_fragments<DIAG, SELF, S, SD>(jvB, jheld, keep, table, dtab, lane, self_lane);
                double2 c_[S + 2], m[S], q[S];
#pragma unroll
                for (int k = 0; k < S + 2; ++k) c_[k] = lds_rec(t0 + (uint32_t)(k - 1) * R);
#pragma unroll
                for (int s = 0; s < S; ++s) m[s] = lds_rec(tm + (uint32_t)s * R);
#pragma unroll
                for (int s = 0; s < S; ++s) q[s] = lds_rec(tp + (uint32_t)s * R);
#pragma unroll
                for (int s = 0; s < S; ++s) {
                    double yr, yi;
                    row_product<DIAG, SD>(c_[1 + s], m[s], c_[s], c_[2 + s], q[s], SELF ? fsB[s] : keep[s][0], keep[s], yr, yi);
                    finish_b(s, yr, yi, c_[1 + s]);
                }
            }
            jvB = jvA;
            jvA = jnext;
            jnext = jn2;
#pragma unroll
            for (int s = 0; s < S; ++s) fsB[s] = fsA[s], fsA[s] = fsN[s];
        }
        cnt += (uint32_t)n_planes;
    }
    if (LISTED) {
        if (panel >= 0)
            flush_dots<NW, 8>(d0, d1, d2, d3, pair_smem, run, wk.lists.panel_runs[panel], wk.lists.panel_runs[panel + 1], panel, n_panels, partials, tickets,
                              dots_step);
    } else {
        const int p = (int)blockIdx.y, r0 = p * (int)gridDim.x;
        flush_dots<NW, 8>(d0, d1, d2, d3, pair_smem, r0 + (int)blockIdx.x, r0, r0 + (int)gridDim.x, p, n_panels, partials, tickets, dots_step);
    }
}

template <bool LISTED> PairKernel pick_pair(bool diag, bool self, bool t2, bool sd) {
    if (sd && !diag) {  // general hopping blocks, real-diagonal on-site blocks
        if (self) return t2 ? cheb_pair_step<false, true, 1, true, LISTED> : cheb_pair_step<false, true, 0, true, LISTED>;
        return t2 ? cheb_pair_step<false, false, 1, true, LISTED> : cheb_pair_step<false, false, 0, true, LISTED>;
    }
    if (self) {
        if (t2) return diag ? cheb_pair_step<true, true, 1, false, LISTED> : cheb_pair_step<false, true, 1, false, LISTED>;
        return diag ? cheb_pair_step<true, true, 0, false, LISTED> : cheb_pair_step<false, true, 0, false, LISTED>;
    }
    if (t2) return diag ? cheb_pair_step<true, false, 1, false, LISTED> : cheb_pair_step<false, false, 1, false, LISTED>;
    return diag ? cheb_pair_step<true, false, 0, false, LISTED> : cheb_pair_step<false, false, 0, false, LISTED>;
}

constexpr int kPairThreads = kPairWarps * 32;
// Dynamic shared memory of cheb_pair_step: the T_n ring, the T_{n+1} ring, two guard records, kRingN + 1 mbarriers.
constexpr size_t kPairSmem = ((size_t)kRingN * (kPairWarps * kPairSites + 2) + (size_t)kRing * kPairWarps * kPairSites + 2) * kRecBytes +
                             8 * (kRingN + 1);

}  // namespace

// The two-step kernel of the current recursion (Pair or EvenPlane) with its patch size, segment length and grid.
int pair_configure(bdg_system *sys, const PlanSwitches &sw) {
    ChebState &st = sys->cheb;
    const EllDev &e = sys->ell;
    const bool diag = st.kernel == BDG_KERNEL_DICT_DIAG, even = st.stepping == Stepping::EvenPlane;
    // On-site fragments per row straight from the table (SELF) when the dictionary is large: then the on-site blocks
    // differ from site to site (disorder, a self-consistent gap, a phase winding) and holding them in registers from
    // plane to plane would reload them on every row through the slow path.
    st.onsite_per_row = sw.pair_self >= 0 ? sw.pair_self != 0 : e.n_unique > 64;
    // Real-diagonal on-site blocks next to general hopping blocks: two multiplications instead of two MMAs
    st.onsite_diag = e.self_diag_usable && !e.diag_usable && sw.ell_sd;
    const PairKernel classic = pick_pair<false>(diag, st.onsite_per_row, even, st.onsite_diag);
    // (the occupancy query counts kPairSmem against the kernel's limit, so the limit is raised first)
    BDG_CUDA(cudaFuncSetAttribute(classic, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPairSmem));
    int per_sm = 1;
    BDG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, classic, kPairThreads, kPairSmem));
    per_sm = std::max(per_sm, 1);
    const int64_t all_slots = (int64_t)sys->sm_count * per_sm;
    const int64_t slots = std::max<int64_t>(1, all_slots / st.n_panels);
    PairWalk &w = st.pair_walk;
    w.Lx = sys->cubic[0];
    w.M = e.pair_M;
    const int p_max = kPairWarps * kPairSites - 2;
    w.open = e.pair_open && sw.pair_open ? 1 : 0;
    const int to_cover = std::max(1, w.M - 2 * w.open);  // n patches own n P (+ 2: the rim sites of a plane with open ends) sites
    const int n_patches_min = (int)ceil_div(to_cover, p_max);
    w.P = sw.pair_p > 0 ? std::min(sw.pair_p, p_max) : (int)ceil_div(to_cover, n_patches_min);  // balanced patches
    w.n_patches = (int)ceil_div(to_cover, w.P);
    // Segment length: every item recomputes one plane of T_{n+1} on either side of its segment and
    // starts with a cold pipeline (about two more plane times); many items balance the CTAs.
    double best = -1.0;
    const int forced = sw.pair_seg;
    for (int n_seg = 1; n_seg <= std::max(1, w.Lx / 4); ++n_seg) {
        const int len = forced > 0 ? std::min(forced, w.Lx) : (int)ceil_div(w.Lx, n_seg);
        const int64_t segs = ceil_div(w.Lx, len);
        const int64_t items = (int64_t)w.n_patches * segs;
        const double balance = (double)items / (double)(ceil_div(items, slots) * slots);
        const double score = balance * len / (len + 4.0);
        if (score > best) {
            best = score;
            w.seg_len = len;
            w.n_segs = (int)segs;
            w.n_items = (int)items;
        }
        if (forced > 0) break;
    }
    constexpr int kPieceCost = 6;  // iterations a piece costs beyond its planes: two halo planes either side, cold pipeline
    BDG_TRY(choose_work_plan(sys, st.work_items, st.n_panels, w.n_patches, w.Lx, w.seg_len, w.n_items, all_slots, kPieceCost, 1.08,
                             sw.pair_balance, w.lists));
    const bool listed = w.lists.pieces != nullptr;
    const PairKernel k = listed ? pick_pair<true>(diag, st.onsite_per_row, even, st.onsite_diag) : classic;
    if (listed) BDG_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPairSmem));
    st.two_step = {k, dim3((unsigned)w.lists.n_ctas, listed ? 1u : (unsigned)st.n_panels), kPairThreads, kPairSmem};
    st.partial_runs = std::max(st.partial_runs, (int)ceil_div(w.lists.n_runs, st.n_panels));
    return BDG_OK;
}

// Pair mode: T_{n+1} -> x_next1, T_{n+2} -> x_next2 and the dot products of both steps (dots_step: 4 rows).
int pair_launch(bdg_system *sys, const void *x_prev, const void *x_cur, void *x_next1, void *x_next2, double *dots_step) {
    ChebState &st = sys->cheb;
    const EllDev &e = sys->ell;
    const Launch<PairKernel> &l = st.two_step;
    note_launch(st, reinterpret_cast<const void *>(l.fn));
    l.fn<<<l.grid, l.threads, l.smem, sys->stream>>>(
        e.dcode.as<int32_t>(), e.table.as<double>(), e.dtab.as<double>(), static_cast<const double2 *>(x_prev),
        static_cast<const double2 *>(x_cur), static_cast<double2 *>(x_next1), static_cast<double2 *>(x_next2),
        (int)e.n_sites, st.n_panels, 2.0 / st.scale, 0.0, 0.0, 0, st.partials.as<double>(), st.tickets.as<unsigned>(), dots_step,
        st.pair_walk);
    BDG_CUDA(cudaGetLastError());
    return BDG_OK;
}

// EvenPlane: E_{j+1} = 2 T_2(H~) E_j - E_{j-1} written over E_{j-1} (x_io); first: E_1 = T_2(H~) E_0.
int t2_launch(bdg_system *sys, bool first, const void *x_cur, void *x_io, double *dots_step) {
    ChebState &st = sys->cheb;
    const EllDev &e = sys->ell;
    const Launch<PairKernel> &l = st.two_step;
    note_launch(st, reinterpret_cast<const void *>(l.fn));
    l.fn<<<l.grid, l.threads, l.smem, sys->stream>>>(
        e.dcode.as<int32_t>(), e.table.as<double>(), e.dtab.as<double>(), static_cast<const double2 *>(x_io),
        static_cast<const double2 *>(x_cur), nullptr, static_cast<double2 *>(x_io), (int)e.n_sites, st.n_panels,
        1.0 / st.scale, (first ? 2.0 : 4.0) / st.scale, first ? 1.0 : 2.0, first ? 1 : 0, st.partials.as<double>(), st.tickets.as<unsigned>(),
        dots_step, st.pair_walk);
    BDG_CUDA(cudaGetLastError());
    return BDG_OK;
}
