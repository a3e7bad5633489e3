// Two applications of H~ per pass over the vectors on THREE-DIMENSIONAL lattices: the even-vector recursion of
// cheb_pair.cu (MODE 1, "T2")
//
//     E_j = T_2j(H~) x,    E_{j+1} = 2 T_2(H~) E_j - E_{j-1} = 4 H~ (H~ E_j) - 2 E_j - E_{j-1}
//
// for cubic lattices with Ly, Lz >= 2 (BASELINE config C4: 64^3).  One launch reads E_j and E_{j-1} and writes E_{j+1}:
// three vector passes for two applications of H~, the intermediate u = H~ E_j lives in shared memory only.
//
// What is different from the kernel for one-dimensional x-planes.  The x-plane is two-dimensional, so a CTA owns a
// PY x PZ patch of it and the halo is a ring, not two sites: u is needed one site around the patch, E_j two sites
// around it.  A 512-byte site record (8 columns) leaves room for 32 sites per plane in 227 KB of shared memory -- a
// 4 x 4 patch would own 2 x 2 -- so this kernel works on FOUR-column panels (256-byte records, ChebState::panel_width = 4)
// and a warp handles two z-adjacent sites at a time: lanes 0..15 the 16 elements (column, component) of the first, lanes
// 16..31 of the second.  That is still one conflict-free 128-bit access per operand (two adjacent records = 512
// contiguous bytes), and still the transposed FP64-MMA formulation: the A fragment of mma.m8n8k4 is the two records
// (row = site half x column), the B fragment the on-site block in fragment order, the C fragment lands in the lane
// that loaded the element.  Two sites share one MMA pair when their on-site blocks have the same dictionary code (the
// bulk of any lattice model); when they differ each gets its own pair and every lane keeps its half.
//
// Matrix: block dictionary with real-diagonal hopping blocks (cheb_ell.cu: DICT + DIAG; the on-site block is any 4x4
// block), open nearest-neighbour stencil, at most kCubeMaxUnique = 64 distinct blocks (fragments are held in registers and
// reloaded when a code changes).  dcode[site][kCubeCodes] holds the dictionary codes towards (self, x-1, y-1, z-1, z+1,
// y+1, x+1) = ascending block column, so that the sums are those of the single-step kernel in the same order.  kNoBlock =
// no block (zero coefficient); kNoSite = "no lattice site there in y / z": the operand is a shared-memory record that
// is never written (rings are cleared per item, copies and stores skip what is outside the lattice), so the held
// coefficient is kept and a patch on the lattice boundary runs without reloading fragments.
//
// An item = (patch, segment [x0, x0 + len) of x).  Iteration i = 0 .. len + 1, planes t <-> x = x0 - 2 + t of E_j in a ring
// of NE planes of (PY + 4) x (PZ + 4) records, staged by bulk async copies (one per y-row, issued by the lanes of warp 0,
// completion on one mbarrier per ring slot):
//   [A] u(x0 - 1 + i) on the patch and its halo ring (corners left out) from E_j planes t = i, i + 1, i + 2
//       -> ring of three u planes of (PY + 2) x (PZ + 2) records; <E_j,E_j>, <u,E_j> on owned sites of owned planes
//   __syncthreads
//   [B] E_{j+1}(x0 - 2 + i), i >= 2, on the owned sites from the three u planes, E_j (ring, t = i) and E_{j-1} (global,
//       loaded one iteration ahead by the thread that overwrites it); <E_{j+1},E_j>, <E_{j+1},u>
//   __syncthreads; plane t = i is dead: its slot takes plane t = i + NE
// Halo values of u (the ring around the patch, one plane either side of the segment) are recomputed, not exchanged.
// The four dot products are reduced like cheb_pair.cu's (fixed order, bit-reproducible) and leave the same rows,
// so cheb.cu's t2_normalize and everything behind it are unchanged.
#include <algorithm>
#include <cstdlib>

#include "bdg_internal.h"
#include "cheb_device.cuh"
#include "cheb_plan.h"
#include "cheb_smem.cuh"
#include "work_lists.h"

namespace {

constexpr int kRec4 = 256;     // one site record at PW = 4: 4 columns x 4 components x complex128
constexpr int kRingU = 3;      // planes of the u ring

__device__ __forceinline__ void mbar_arrive_plain(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(bar) : "memory");
}

// Fragments of the two sites a warp works on, held from body to body and reloaded when a code differs from the held
// one.  Lane s * 8 + u (s = 0, 1; u = 0..6) carries the code of site s, direction u.
struct Held {
    double b0 = 0.0, b1 = 0.0;  // on-site B fragment (this lane's double) of site 0 / site 1
    double h[7] = {0, 0, 0, 0, 0, 0, 0};  // h[u]: this lane's diagonal entry of its site's hopping block towards u (u >= 1)
    int jheld = -3;
    bool two = false;           // the two sites have different on-site blocks
};

// The reload path is taken a few times per item, but its loads would share a scoreboard with the prefetches issued at the
// top of every iteration (ptxas has six): the first MMA after the branch then waits for those prefetches -- a full HBM
// latency per iteration (ncu: 17 % of all stall samples on that one instruction, profiles/r02/24_cube_c4k8_v1_hot_instructions.txt).
// An integer operation on the loaded value INSIDE the branch waits there instead, and what leaves the branch is the result
// of a fixed-latency instruction.
__device__ __forceinline__ double settle(double v, int n_panels /* > 0: the XOR mask is a zero the compiler cannot see through */) {
    return __longlong_as_double(__double_as_longlong(v) ^ (long long)(n_panels >> 30));
}

__device__ __forceinline__ void hold_cube(int jv, Held &H, const double *__restrict__ table, const double *__restrict__ dtab,
                                          int lane, int n_panels) {
    const bool code_lane = lane < 16 && (lane & 7) < 7;
    const unsigned changed = __ballot_sync(kFull, code_lane && jv != H.jheld && jv != kNoSite);
    if (changed) {
        if (code_lane && jv != kNoSite) H.jheld = jv;
        const bool upper = lane >= 16;
        if (changed & 0x0101u) {
            const int c0 = __shfl_sync(kFull, H.jheld, 0), c1 = __shfl_sync(kFull, H.jheld, 8);
            H.b0 = settle(c0 >= 0 ? __ldg(table + (size_t)c0 * 32 + lane) : 0.0, n_panels);
            H.b1 = settle(c1 >= 0 ? __ldg(table + (size_t)c1 * 32 + lane) : 0.0, n_panels);
            H.two = c0 != c1;
        }
#pragma unroll
        for (int u = 1; u < 7; ++u) {
            if (changed & (0x0101u << u)) {
                const int c0 = __shfl_sync(kFull, H.jheld, u), c1 = __shfl_sync(kFull, H.jheld, 8 + u);
                const int c = upper ? c1 : c0;
                H.h[u] = settle(c >= 0 ? __ldg(dtab + (size_t)c * 4 + (lane & 3)) : 0.0, n_panels);
            }
        }
    }
}

// y = sum_u B_u x_u for this lane's element: on-site block by two FP64 MMAs (four when the two sites differ), the six
// real-diagonal hopping blocks by two DFMA each, in ascending block column (x-1, y-1, z-1, z+1, y+1, x+1).
__device__ __forceinline__ void onsite_product(const double2 &c, const Held &H, bool upper, double &yr, double &yi) {
    double a10 = 0.0, a11 = 0.0, a20 = 0.0, a21 = 0.0;
    dmma_8x8x4(a10, a11, c.x, H.b0);
    dmma_8x8x4(a20, a21, c.y, H.b0);
    if (H.two) {
        double e10 = 0.0, e11 = 0.0, e20 = 0.0, e21 = 0.0;
        dmma_8x8x4(e10, e11, c.x, H.b1);
        dmma_8x8x4(e20, e21, c.y, H.b1);
        if (upper) a10 = e10, a11 = e11, a20 = e20, a21 = e21;
    }
    yr = a10 - a21;
    yi = a11 + a20;
}
__device__ __forceinline__ void hop(const double2 &x, double b, double &yr, double &yi) {
    yr = fma(b, x.x, yr);
    yi = fma(b, x.y, yi);
}

// NW warps, one CTA per SM.  Body lists (one body = two z-adjacent sites): [A] the u region = the patch and its halo
// ring without the corners -- rows 0 and PY + 1 of the region hold PZ / 2 bodies, the PY rows between (PZ + 2) / 2 --,
// [B] the PY x PZ / 2 owned bodies; body b goes to warp b % NW.  At PY = PZ = 8, NW = 16: 48 + 32 bodies, three + two per warp.
// LISTED: the pieces come from the work lists of CubeWalk (balanced plan, grid = (n_ctas, 1)), else from the item index
// (classic plan, grid = (CTAs per panel, panels)).
template <int NW, int PY, int PZ, int NE, bool LISTED = false>
__global__ void __launch_bounds__(NW * 32, 1)
cheb_cube_step(const int32_t *__restrict__ dcode, const double *__restrict__ table, const double *__restrict__ dtab,
               const double2 *__restrict__ xb /* E_j */, double2 *__restrict__ xio /* E_{j-1} -> E_{j+1} */, int n_sites,
               int n_panels, double alpha, double alpha2, double csub, int first, double *__restrict__ partials,
               unsigned *__restrict__ tickets, double *__restrict__ dots_step, const CubeWalk wk) {
    static_assert(PZ % 2 == 0 && PY + 4 <= 32, "bodies are z-pairs; one lane of warp 0 stages one row of a plane");
    constexpr int EY = PY + 4, EZ = PZ + 4, UY = PY + 2, UZ = PZ + 2, R = kRec4;
    constexpr uint32_t PLANE_E = EY * EZ * R, PLANE_U = UY * UZ * R;
    constexpr int HZ = PZ / 2, MZ = UZ / 2;
    constexpr int NA = 2 * HZ + PY * MZ, NB = PY * HZ;
    constexpr int RA = (NA + NW - 1) / NW, RB = (NB + NW - 1) / NW;
    static_assert(NA >= NW && NB >= 1, "every warp has a first [A] body (it waits for the newest plane there)");
    extern __shared__ __align__(128) unsigned char cube_smem[];
    const uint32_t sE = smem_u32(cube_smem);      // E_j planes, local site (ly, lz) = (y - (y0 - 2), z - (z0 - 2))
    const uint32_t sU = sE + NE * PLANE_E;        // u planes, local site (y - (y0 - 1), z - (z0 - 1))
    const uint32_t sBar = sU + kRingU * PLANE_U;  // one mbarrier per E_j slot

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool upper = lane >= 16;
    const int half = lane >> 4;
    int panel = -1, run = -1;  // LISTED: the panel of the pieces in hand, their run

    if (threadIdx.x == 0) {
#pragma unroll
        for (int r = 0; r < NE; ++r) mbar_init(sBar + 8 * r, 1);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    uint32_t cnt = 0;  // E_j planes consumed by the items before this one
    const int plane_sites = wk.Ly * wk.Lz;
    double d0 = 0.0, d1 = 0.0, d2 = 0.0, d3 = 0.0;
    Held H;

    // ---- this warp's bodies: shared-memory offsets (the same for every item) ------------------------------------
    uint32_t aE[RA], aU[RA];  // [A]: own records in an E_j plane / in a u plane (+ this lane's 16 bytes)
    int aly[RA], alz[RA];     // ... and their position in the u region (first site of the pair)
    uint32_t bE[RB], bU[RB];  // [B]: likewise
    int boy[RB], boz[RB];     // ... position in the patch
#pragma unroll
    for (int r = 0; r < RA; ++r) {
        const int b = warp + NW * r;
        int ly = 0, lz = 1;
        if (b < HZ) ly = 0, lz = 1 + 2 * b;
        else if (b < HZ + PY * MZ) ly = 1 + (b - HZ) / MZ, lz = 2 * ((b - HZ) % MZ);
        else ly = UY - 1, lz = 1 + 2 * (b - HZ - PY * MZ);
        if (b >= NA) ly = 1, lz = 0;  // idle slot: any valid position (never executed)
        aly[r] = ly, alz[r] = lz;
        aE[r] = (uint32_t)((ly + 1) * EZ + lz + 1) * R + (uint32_t)lane * 16u;
        aU[r] = (uint32_t)(ly * UZ + lz) * R + (uint32_t)lane * 16u;
    }
#pragma unroll
    for (int r = 0; r < RB; ++r) {
        const int b = min(warp + NW * r, NB - 1);
        boy[r] = b / HZ, boz[r] = 2 * (b % HZ);
        bU[r] = (uint32_t)((boy[r] + 1) * UZ + boz[r] + 1) * R + (uint32_t)lane * 16u;
        bE[r] = (uint32_t)((boy[r] + 2) * EZ + boz[r] + 2) * R + (uint32_t)lane * 16u;
    }
    const bool code_lane = lane < 16 && (lane & 7) < 7;
    const int cs = lane >> 3, cu = lane & 7;  // code lanes: site of the pair, direction

    const int item0 = LISTED ? wk.lists.cta_begin[blockIdx.x] : (int)blockIdx.x, item1 = LISTED ? wk.lists.cta_begin[blockIdx.x + 1] : wk.n_items;
    for (int item = item0; item < item1; item += LISTED ? 1 : (int)gridDim.x) {
        int4 piece;  // panel, patch, x0, len
        if (LISTED) {
            piece = wk.lists.pieces[item];  // (run, patch, x0, len)
            if (piece.x != run) {
                if (run >= 0) {
                    flush_dots<NW, 4>(d0, d1, d2, d3, cube_smem, run, wk.lists.panel_runs[panel], wk.lists.panel_runs[panel + 1], panel, n_panels, partials,
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
        const size_t pbase = (size_t)piece.x * n_sites * 16;
        const double2 *const tb = xb + pbase;
        double2 *const tio = xio + pbase;
        const int patch = piece.y;
        const int py = patch / wk.nPz, pz = patch - py * wk.nPz;
        const int y0 = py * PY, z0 = pz * PZ;
        const int x0 = piece.z, len = piece.w;
        const int n_planes = len + 4;  // E_j planes x0 - 2 .. x0 + len + 1; those outside the lattice are not copied

        __syncthreads();  // every warp is done with the previous item's planes (all of them were waited for)
        for (uint32_t o = threadIdx.x * 16u; o < NE * PLANE_E + kRingU * PLANE_U; o += NW * 32 * 16u)
            sts_rec(sE + o, make_double2(0.0, 0.0));
        asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");  // the clears are ordered before the bulk copies
        __syncthreads();

        // Row `lane` of a plane (warp 0): y = y0 - 2 + lane, z from max(z0 - 2, 0) to min(z0 + PZ + 2, Lz)
        uint32_t row_dst = 0, row_bytes = 0, plane_bytes = 0;
        size_t row_src = 0;
        if (warp == 0) {
            const int y = y0 - 2 + lane;
            const int zlo = max(z0 - 2, 0), zhi = min(z0 + PZ + 2, wk.Lz);
            if (lane < EY && y >= 0 && y < wk.Ly && zhi > zlo) {
                row_bytes = (uint32_t)(zhi - zlo) * R;
                row_dst = (uint32_t)(lane * EZ + zlo - (z0 - 2)) * R;
                row_src = ((size_t)y * wk.Lz + zlo) * 16;
            }
            plane_bytes = row_bytes;
#pragma unroll
            for (int d = 16; d; d >>= 1) plane_bytes += __shfl_xor_sync(kFull, plane_bytes, d);
        }
        auto issue = [&](int t) {
            if (warp == 0 && t < n_planes) {
                const int x = x0 - 2 + t;
                const uint32_t c = cnt + (uint32_t)t, r = c % NE;
                const uint32_t bar = sBar + 8 * r;
                const bool inside = x >= 0 && x < wk.Lx && plane_bytes > 0;
                if (lane == 0) {
                    if (inside) mbar_expect_tx(bar, plane_bytes);
                    else mbar_arrive_plain(bar);
                }
                __syncwarp();
                if (inside && row_bytes) bulk_g2s(sE + r * PLANE_E + row_dst, tb + (size_t)x * plane_sites * 16 + row_src, row_bytes, bar);
            }
        };
        auto wait = [&](int t) {
            if (t < n_planes) {
                const uint32_t c = cnt + (uint32_t)t;
                mbar_wait(sBar + 8 * (c % NE), (c / NE) & 1u);
            }
        };
        for (int t = 0; t < NE; ++t) issue(t);

        // ---- item-dependent part of the body descriptors --------------------------------------------------------
        bool existA[RA], ownA[RA], existB[RB];
        int codeA[RA], codeB[RB];  // code lanes: offset of (site, direction) inside a plane of dcode, -1 = no such site
        ptrdiff_t gB[RB];          // [B]: element of the pair inside a plane of the vectors
#pragma unroll
        for (int r = 0; r < RA; ++r) {
            const int y = y0 - 1 + aly[r], zf = z0 - 1 + alz[r];
            const bool row_ok = warp + NW * r < NA && y >= 0 && y < wk.Ly;
            existA[r] = row_ok && zf + half >= 0 && zf + half < wk.Lz;
            ownA[r] = existA[r] && aly[r] >= 1 && aly[r] <= PY && alz[r] + half >= 1 && alz[r] + half <= PZ;
            const int zs = zf + cs;
            codeA[r] = code_lane && row_ok && zs >= 0 && zs < wk.Lz ? (y * wk.Lz + zs) * kCubeCodes + cu : -1;
        }
#pragma unroll
        for (int r = 0; r < RB; ++r) {
            const int y = y0 + boy[r], zf = z0 + boz[r];
            const bool row_ok = warp + NW * r < NB && y < wk.Ly;
            existB[r] = row_ok && zf + half < wk.Lz;
            const int zs = zf + cs;
            codeB[r] = code_lane && row_ok && zs < wk.Lz ? (y * wk.Lz + zs) * kCubeCodes + cu : -1;
            gB[r] = ((ptrdiff_t)y * wk.Lz + zf) * 16 + lane;
        }
        // codes of the plane of [A] in this / the next iteration, of the plane of [B] likewise (loaded one iteration ahead)
        int jA[RA], jAn[RA], jB[RB], jBn[RB];
        {
            const int xa = x0 - 1;
            const size_t po = (size_t)max(xa, 0) * plane_sites * kCubeCodes;
#pragma unroll
            for (int r = 0; r < RA; ++r) {
                jA[r] = jAn[r] = kNoSite;
                if (xa >= 0 && codeA[r] >= 0) jA[r] = __ldg(dcode + po + codeA[r]);
            }
#pragma unroll
            for (int r = 0; r < RB; ++r) jB[r] = jBn[r] = kNoSite;
        }
        double2 pv[RB], pvn[RB];  // E_{j-1} of the plane of [B] in this / the next iteration
#pragma unroll
        for (int r = 0; r < RB; ++r) pv[r] = pvn[r] = make_double2(0.0, 0.0);
        wait(0);
        wait(1);

        for (int i = 0; i <= len + 1; ++i) {
            const int xa = x0 - 1 + i;  // plane of [A]; [B] works on xa - 1
            const bool a_valid = xa >= 0 && xa < wk.Lx;
            const bool store = i >= 1 && i <= len;  // xa is an owned plane
            // one iteration ahead: codes of the next planes, E_{j-1} of the plane [B] overwrites next
            {
                const int xn = xa + 1;
                const bool n_valid = i <= len && xn >= 0 && xn < wk.Lx;
                const size_t pn = (size_t)(n_valid ? xn : 0) * plane_sites * kCubeCodes;
                const size_t pa = (size_t)(a_valid ? xa : 0) * plane_sites * kCubeCodes;
#pragma unroll
                for (int r = 0; r < RA; ++r) {
                    jAn[r] = kNoSite;
                    if (n_valid && codeA[r] >= 0) jAn[r] = __ldg(dcode + pn + codeA[r]);
                }
#pragma unroll
                for (int r = 0; r < RB; ++r) {
                    jBn[r] = kNoSite;
                    if (store && codeB[r] >= 0) jBn[r] = __ldg(dcode + pa + codeB[r]);
                    pv[r] = pvn[r];
                    if (store && existB[r] && !first) pvn[r] = ld_prev_rw(tio + (ptrdiff_t)xa * plane_sites * 16 + gB[r]);
                }
            }
            const uint32_t c = cnt + (uint32_t)i;
            const uint32_t eM = sE + (c % NE) * PLANE_E, eC = sE + ((c + 1) % NE) * PLANE_E, eP = sE + ((c + 2) % NE) * PLANE_E;
            const uint32_t uW = sU + (uint32_t)(i % kRingU) * PLANE_U;
            // ---- [A] ------------------------------------------------------------------------------------------
            if (a_valid) {
#pragma unroll
                for (int r = 0; r < RA; ++r) {
                    if (warp + NW * r < NA) {
                        hold_cube(jA[r], H, table, dtab, lane, n_panels);
                        const uint32_t a = eC + aE[r];
                        const double2 own = lds_rec(a), xm = lds_rec(eM + aE[r]), ym = lds_rec(a - EZ * R), zm = lds_rec(a - R);
                        const double2 zp = lds_rec(a + R), yp = lds_rec(a + EZ * R);
                        double yr, yi;
                        onsite_product(own, H, upper, yr, yi);
                        hop(xm, H.h[1], yr, yi);
                        hop(ym, H.h[2], yr, yi);
                        hop(zm, H.h[3], yr, yi);
                        hop(zp, H.h[4], yr, yi);
                        hop(yp, H.h[5], yr, yi);
                        if (r == 0) wait(i + 2);  // the newest plane feeds the last term only
                        const double2 xp = lds_rec(eP + aE[r]);
                        hop(xp, H.h[6], yr, yi);
                        const double2 u = make_double2(alpha * yr, alpha * yi);
                        if (existA[r]) sts_rec(uW + aU[r], u);
                        if (store && ownA[r]) {
                            d0 = fma(own.x, own.x, fma(own.y, own.y, d0));
                            d1 = fma(u.x, own.x, fma(u.y, own.y, d1));
                        }
                    }
                }
            } else {
                wait(i + 2);
            }
            __syncthreads();  // u of this plane complete in the ring
            // ---- [B] ------------------------------------------------------------------------------------------
            if (i >= 2) {
                const uint32_t uM = sU + (uint32_t)((i - 2) % kRingU) * PLANE_U, uC = sU + (uint32_t)((i - 1) % kRingU) * PLANE_U;
                double2 *pout = tio + (ptrdiff_t)(xa - 1) * plane_sites * 16;
#pragma unroll
                for (int r = 0; r < RB; ++r) {
                    if (warp + NW * r < NB) {
                        hold_cube(jB[r], H, table, dtab, lane, n_panels);
                        const uint32_t a = uC + bU[r];
                        const double2 own = lds_rec(a), xm = lds_rec(uM + bU[r]), ym = lds_rec(a - UZ * R), zm = lds_rec(a - R);
                        const double2 zp = lds_rec(a + R), yp = lds_rec(a + UZ * R), xp = lds_rec(uW + bU[r]);
                        const double2 t = lds_rec(eM + bE[r]);  // E_j of the row
                        double yr, yi;
                        onsite_product(own, H, upper, yr, yi);
                        hop(xm, H.h[1], yr, yi);
                        hop(ym, H.h[2], yr, yi);
                        hop(zm, H.h[3], yr, yi);
                        hop(zp, H.h[4], yr, yi);
                        hop(yp, H.h[5], yr, yi);
                        hop(xp, H.h[6], yr, yi);
                        const double2 sub = make_double2(fma(csub, t.x, pv[r].x), fma(csub, t.y, pv[r].y));
                        const double2 out = make_double2(fma(alpha2, yr, -sub.x), fma(alpha2, yi, -sub.y));
                        if (existB[r]) {
                            pout[gB[r]] = out;
                            d2 = fma(out.x, t.x, fma(out.y, t.y, d2));
                            d3 = fma(out.x, own.x, fma(out.y, own.y, d3));
                        }
                    }
                }
            }
            __syncthreads();  // plane t = i and the oldest u plane are dead
            issue(i + NE);
#pragma unroll
            for (int r = 0; r < RA; ++r) jA[r] = jAn[r];
#pragma unroll
            for (int r = 0; r < RB; ++r) jB[r] = jBn[r];
        }
        cnt += (uint32_t)n_planes;
    }

    if (LISTED) {
        if (panel >= 0)
            flush_dots<NW, 4>(d0, d1, d2, d3, cube_smem, run, wk.lists.panel_runs[panel], wk.lists.panel_runs[panel + 1], panel, n_panels, partials, tickets,
                              dots_step);
    } else {
        const int p = (int)blockIdx.y, r0 = p * (int)gridDim.x;
        flush_dots<NW, 4>(d0, d1, d2, d3, cube_smem, r0 + (int)blockIdx.x, r0, r0 + (int)gridDim.x, p, n_panels, partials, tickets, dots_step);
    }
}

struct CubeShape {
    int warps, py, pz, ne;
    int rounds;  // bodies per warp and iteration ([A] + [B])
    CubeKernel kernel, listed;  // classic plan / balanced plan (work lists)
    size_t smem;
};

template <int NW, int PY, int PZ, int NE> CubeShape make_shape() {
    CubeShape s;
    s.warps = NW, s.py = PY, s.pz = PZ, s.ne = NE;
    constexpr int NA = PZ + PY * (PZ + 2) / 2, NB = PY * PZ / 2;
    s.rounds = (NA + NW - 1) / NW + (NB + NW - 1) / NW;
    s.kernel = cheb_cube_step<NW, PY, PZ, NE>;
    s.listed = cheb_cube_step<NW, PY, PZ, NE, true>;
    s.smem = (size_t)NE * (PY + 4) * (PZ + 4) * kRec4 + (size_t)kRingU * (PY + 2) * (PZ + 2) * kRec4 + 8 * NE;
    return s;
}

constexpr int kCubeShapes = 3;
CubeShape cube_shape(int which) {
    switch (which) {
        case 1: return make_shape<16, 6, 8, 5>();   // two planes of copy lead
        case 2: return make_shape<16, 4, 8, 6>();   // small planes: three planes of lead, 28 + 16 bodies
        default: return make_shape<16, 8, 8, 4>();  // 48 + 32 bodies = exactly three + two per warp
    }
}

}  // namespace

// Patch shape, segment length and grid for the current recursion: the plan with the fewest body rounds on the
// critical path (waves x planes per item x bodies per warp and plane).
int cube_configure(bdg_system *sys, const PlanSwitches &sw) {
    ChebState &st = sys->cheb;
    const int Lx = sys->cubic[0], Ly = sys->cubic[1], Lz = sys->cubic[2];
    const int64_t slots = std::max<int64_t>(1, (int64_t)sys->sm_count / st.n_panels);
    double best = -1.0;
    int chosen = 0;
    for (int which = 0; which < kCubeShapes; ++which) {
        if (sw.cube_shape >= 0 && which != sw.cube_shape) continue;
        const CubeShape shape = cube_shape(which);
        const int nPy = (int)ceil_div(Ly, shape.py), nPz = (int)ceil_div(Lz, shape.pz);
        const int64_t patches = (int64_t)nPy * nPz;
        for (int n_seg = 1; n_seg <= std::max(1, Lx / 4); ++n_seg) {
            const int len = sw.cube_seg > 0 ? std::min(sw.cube_seg, Lx) : (int)ceil_div(Lx, n_seg);
            const int64_t segs = ceil_div(Lx, len), items = patches * segs;
            const double cost = (double)ceil_div(items, slots) * (len + 4.0) * shape.rounds;
            if (best < 0.0 || cost < best) {
                best = cost;
                CubeWalk &w = st.cube_walk;
                w.Lx = Lx, w.Ly = Ly, w.Lz = Lz;
                w.nPy = nPy, w.nPz = nPz, w.n_patches = (int)patches;
                w.seg_len = len, w.n_segs = (int)segs, w.n_items = (int)items;
                chosen = which;
            }
            if (sw.cube_seg > 0) break;
        }
    }
    CubeWalk &w = st.cube_walk;
    // Balanced plan: one contiguous chunk of the (panel, patch, x) space per SM instead of whole patch columns -- C4 with 8
    // columns is 128 columns of 64 planes on 148 SMs.
    constexpr int kPieceCost = 6;
    BDG_TRY(choose_work_plan(sys, st.work_items, st.n_panels, w.n_patches, Lx, w.seg_len, w.n_items, sys->sm_count, kPieceCost, 1.0,
                             sw.cube_balance, w.lists));
    const CubeShape shape = cube_shape(chosen);
    const bool listed = w.lists.pieces != nullptr;
    const CubeKernel k = listed ? shape.listed : shape.kernel;
    BDG_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)shape.smem));
    st.cube_step = {k, dim3((unsigned)w.lists.n_ctas, listed ? 1u : (unsigned)st.n_panels), (unsigned)shape.warps * 32, shape.smem};
    st.partial_runs = std::max(st.partial_runs, (int)ceil_div(w.lists.n_runs, st.n_panels));
    return BDG_OK;
}

// E_{j+1} = 2 T_2(H~) E_j - E_{j-1} written over E_{j-1} (x_io); first: E_1 = T_2(H~) E_0.  Same contract as t2_launch.
int cube_launch(bdg_system *sys, bool first, const void *x_cur, void *x_io, double *dots_step) {
    ChebState &st = sys->cheb;
    const EllDev &e = sys->ell;
    const Launch<CubeKernel> &l = st.cube_step;
    note_launch(st, reinterpret_cast<const void *>(l.fn));
    l.fn<<<l.grid, l.threads, l.smem, sys->stream>>>(
        e.dcode3.as<int32_t>(), e.table.as<double>(), e.dtab.as<double>(), static_cast<const double2 *>(x_cur),
        static_cast<double2 *>(x_io), (int)e.n_sites, st.n_panels, 1.0 / st.scale, (first ? 2.0 : 4.0) / st.scale, first ? 1.0 : 2.0,
        first ? 1 : 0, st.partials.as<double>(), st.tickets.as<unsigned>(), dots_step, st.cube_walk);
    BDG_CUDA(cudaGetLastError());
    return BDG_OK;
}
