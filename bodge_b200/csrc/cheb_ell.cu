// Chebyshev step on the kernel-native matrix format ("ELL"): fixed-width block rows, diagonal
// block first, blocks stored in MMA B-fragment order.  This is the default step kernel for
// lattice Hamiltonians (every row has <= 8 blocks and almost all rows have the same count);
// ragged / long-row matrices use the generic BSR kernel in cheb.cu.
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

// ---- building the format ----------------------------------------------------------------------
// need[row] = blocks of the row, +1 if the diagonal block is absent (slot 0 is reserved for it)
__global__ void __launch_bounds__(256)
ell_row_need(int n_sites, const int32_t *__restrict__ indptr, const int32_t *__restrict__ indices,
             int *__restrict__ max_need) {
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    int need = 0;
    if (row < n_sites) {
        const int p0 = indptr[row], p1 = indptr[row + 1];
        bool self = false;
        for (int p = p0; p < p1; ++p) self |= indices[p] == row;
        need = p1 - p0 + (self ? 0 : 1);
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) need = max(need, __shfl_xor_sync(0xffffffffu, need, d));
    if ((threadIdx.x & 31) == 0 && need > 0) atomicMax(max_need, need);
}

// One warp per (row, slot); lane l writes double l of the slot in B-fragment order.
__global__ void __launch_bounds__(256)
ell_fill(int n_sites, int width, const int32_t *__restrict__ indptr, const int32_t *__restrict__ indices,
         const double *__restrict__ data, int32_t *__restrict__ cidx, double *__restrict__ cdata) {
    const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= (int64_t)n_sites * width) return;
    const int row = (int)(w / width), slot = (int)(w % width);
    const int p0 = indptr[row], cnt = indptr[row + 1] - p0;
    int self = -1;  // position of the diagonal block inside the row
    for (int t = 0; t < cnt; ++t)
        if (indices[p0 + t] == row) self = t;
    int src;  // position inside the row feeding this slot, or -1
    if (slot == 0) {
        src = self;
    } else {
        src = slot - 1;
        if (self >= 0 && src >= self) src += 1;
        if (src >= cnt) src = -1;
    }
    double v = 0.0;
    if (src >= 0) {
        const int a = lane >> 3, part = (lane >> 2) & 1, b = lane & 3;
        v = data[((size_t)(p0 + src) * 16 + a * 4 + b) * 2 + part];
    }
    cdata[w * 32 + lane] = v;
    if (lane == 0) cidx[w] = src >= 0 ? indices[p0 + src] : row;
}

// ---- block dictionary ---------------------------------------------------------------------------
// Distinct blocks are found with an open-addressing hash table keyed by a 64-bit hash of the
// block's 256 bytes; every slot is then compared bit for bit with its table entry, so a hash
// collision can only disable the format, never change a result.
constexpr unsigned long long kEmptyKey = ~0ull;

// One warp per slot: hash, find-or-insert, remember the table position and the smallest slot id
// holding that key (the representative whose bytes become the table entry).  The table is sized
// for few distinct blocks; when more than `limit` keys have been inserted the pass is abandoned
// (*overflow = 1) and the host retries with a larger table or gives the format up.
__global__ void __launch_bounds__(256)
dict_insert(int64_t n_slots, const double *__restrict__ cdata, unsigned long long *__restrict__ keys,
            int *__restrict__ rep, unsigned cap_mask, int32_t *__restrict__ where, int *__restrict__ counter,
            int limit, int *__restrict__ overflow) {
    const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= n_slots) return;
    const uint64_t bits = (uint64_t)__double_as_longlong(cdata[w * 32 + lane]);
    uint64_t h = mix64(bits + 0x9E3779B97F4A7C15ull * (uint64_t)(lane + 1));
#pragma unroll
    for (int d = 16; d; d >>= 1) h += __shfl_xor_sync(0xffffffffu, h, d);
    h = mix64(h);
    if (h == kEmptyKey) h = 0x1234567ull;
    if (lane != 0) return;
    unsigned pos = (unsigned)h & cap_mask;
    for (;;) {
        unsigned long long seen = *((volatile unsigned long long *)(keys + pos));  // cheap hit for repeated blocks
        if (seen == kEmptyKey) {
            seen = atomicCAS(keys + pos, kEmptyKey, (unsigned long long)h);
            if (seen == kEmptyKey && atomicAdd(counter, 1) >= limit) *overflow = 1;
        }
        if (seen == kEmptyKey || seen == h) break;
        if (*((volatile int *)overflow)) {
            where[w] = 0;
            return;
        }
        pos = (pos + 1) & cap_mask;
    }
    if (*((volatile int *)(rep + pos)) > (int)w) atomicMin(rep + pos, (int)w);
    where[w] = (int32_t)pos;
}

// flag[slot] = 1 iff the slot is the representative of its key (the smallest slot id holding that block).  The
// exclusive scan of the flags numbers the distinct blocks in SLOT order, so the table follows the matrix: the
// on-site blocks of consecutive sites sit next to each other (a kernel that fetches a site-dependent on-site
// block per row then streams the table instead of gathering 256-byte pieces from all over it).
__global__ void __launch_bounds__(256)
dict_flag_reps(int64_t n_slots, const int *__restrict__ rep, const int32_t *__restrict__ where, int32_t *__restrict__ flag) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n_slots) flag[t] = rep[where[t]] == (int)t;
}

// One warp per slot: code = rank of its representative among the representatives (dense[]: scanned flags); the
// representative writes the table entry; everyone else is compared with the representative's bytes.
__global__ void __launch_bounds__(256)
dict_emit(int64_t n_slots, const double *__restrict__ cdata, const int *__restrict__ rep,
          const int32_t *__restrict__ dense, const int32_t *__restrict__ where, int32_t *__restrict__ ccode,
          double *__restrict__ table, int table_cap, int32_t *__restrict__ posid, int *__restrict__ mismatch) {
    const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= n_slots) return;
    const int r = rep[where[w]];
    const int code = dense[r];
    const long long mine = __double_as_longlong(cdata[w * 32 + lane]);
    if (r == (int)w) {
        if (code < table_cap) table[(size_t)code * 32 + lane] = __longlong_as_double(mine);
        if (lane == 0) posid[where[w]] = code;  // hash position -> code: later updates look new blocks up here (ell_patch)
    } else if (mine != __double_as_longlong(cdata[(int64_t)r * 32 + lane])) {
        *mismatch = 1;
    }
    if (lane == 0) ccode[w] = code;
}

// dtab[code][a] = Re of diagonal entry (a, a) of table block `code`; isdiag[code] = the block has
// nothing else (all other real and imaginary parts compare == 0).
__global__ void __launch_bounds__(256)
dict_diag_table(int n_unique, const double *__restrict__ table, double *__restrict__ dtab, int *__restrict__ isdiag) {
    const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (w >= n_unique) return;
    const double v = table[(size_t)w * 32 + lane];
    const int a = lane >> 3, part = (lane >> 2) & 1, b = lane & 3;  // double `lane` = part (re/im) of entry (a, b)
    const bool on_diag = part == 0 && a == b;
    const unsigned other = __ballot_sync(0xffffffffu, !on_diag && v != 0.0);
    if (on_diag) dtab[(size_t)w * 4 + a] = v;
    if (lane == 0) isdiag[w] = other == 0u;
}

// bad[0] = 1 if any slot other than slot 0 holds a block that is not real-diagonal, bad[1] = 1 if any slot 0 does.
__global__ void __launch_bounds__(256)
dict_offsite_diag(int64_t n_slots, int width, const int32_t *__restrict__ ccode, const int *__restrict__ isdiag,
                  int *__restrict__ bad) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_slots) return;
    if (!isdiag[ccode[t]]) bad[t % width == 0 ? 1 : 0] = 1;
}

// ---- incremental update after a scatter (SURVEY 8f-3: re-enter `with`, change a few terms, ask again) -----------
// One warp per touched skeleton block: copy it into its place in `packed`, into its fixed-width slot (fragment
// order), look it up in -- or add it to -- the dictionary and rewrite the slot's code (and direction code).
// status: [0] distinct blocks so far, [1] zero pattern changed, [2] table full, [3] hash collision, [4] an
// off-site block that is not real-diagonal (the DIAG kernels no longer apply), [5] an on-site block that is not (SD).
struct PatchArgs {
    const int32_t *s_indices, *s_brow;
    const double *s_data;
    const int32_t *flags, *pos;
    double *p_data;
    int width;
    const int32_t *cidx;
    double *cdata;
    int32_t *ccode;
    int dict;
    unsigned long long *keys;
    int32_t *posid;
    unsigned cap_mask;
    double *table, *dtab;
    int table_cap, diag_required, self_diag_required;
    int32_t *dcode;
    int Lx, M;
    int32_t *dcode3;
    int Ly, Lz;
    int *status;
};

__global__ void __launch_bounds__(256)
patch_blocks(int64_t n, const int32_t *__restrict__ klist, const PatchArgs a) {
    const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= n) return;
    const int k = klist[w];
    if (k < 0) return;
    const double vs = a.s_data[(size_t)k * 32 + lane];  // skeleton order: (row a, column b, re/im) = double (a*4+b)*2+part
    const bool nz = __ballot_sync(kFull, vs != 0.0) != 0u;
    if (nz != (a.flags[k] != 0)) {
        if (lane == 0) a.status[1] = 1;
        return;
    }
    if (!nz) return;
    a.p_data[(size_t)a.pos[k] * 32 + lane] = vs;
    if (a.width == 0) return;
    const int row = a.s_brow[k], col = a.s_indices[k];
    int u = 0;
    if (col != row) {
        const bool hit = lane >= 1 && lane < a.width && a.cidx[(size_t)row * a.width + lane] == col;
        const unsigned m = __ballot_sync(kFull, hit);
        if (m == 0u) {  // cannot happen for a block that was already stored
            if (lane == 0) a.status[1] = 1;
            return;
        }
        u = __ffs(m) - 1;
    }
    const int64_t slot = (int64_t)row * a.width + u;
    const int fa = lane >> 3, part = (lane >> 2) & 1, fb = lane & 3;  // fragment order (ell_fill)
    const double f = a.s_data[(size_t)k * 32 + (fa * 4 + fb) * 2 + part];
    a.cdata[slot * 32 + lane] = f;
    if (!a.dict) return;
    uint64_t h = mix64((uint64_t)__double_as_longlong(f) + 0x9E3779B97F4A7C15ull * (uint64_t)(lane + 1));
#pragma unroll
    for (int d = 16; d; d >>= 1) h += __shfl_xor_sync(kFull, h, d);
    h = mix64(h);
    if (h == kEmptyKey) h = 0x1234567ull;
    int id = -1, won = 0;
    unsigned pos = 0;
    if (lane == 0) {
        pos = (unsigned)h & a.cap_mask;
        for (;;) {
            unsigned long long seen = *((volatile unsigned long long *)(a.keys + pos));
            if (seen == kEmptyKey) {
                seen = atomicCAS(a.keys + pos, kEmptyKey, (unsigned long long)h);
                if (seen == kEmptyKey) {
                    won = 1;
                    id = atomicAdd(a.status, 1);
                    if (id >= a.table_cap) {
                        a.status[2] = 1;
                        id = -2;
                    }
                    break;
                }
            }
            if (seen == h) break;
            pos = (pos + 1) & a.cap_mask;
        }
        if (!won) {  // someone holds the key: its code is published once the table entry is in place
            while ((id = *((volatile int32_t *)(a.posid + pos))) == -1) {}
        }
    }
    id = __shfl_sync(kFull, id, 0);
    won = __shfl_sync(kFull, won, 0);
    pos = __shfl_sync(kFull, pos, 0);
    const bool on_diag = part == 0 && fa == fb;
    const bool isdiag = __ballot_sync(kFull, !on_diag && f != 0.0) == 0u;
    if (won) {
        if (id >= 0) {
            a.table[(size_t)id * 32 + lane] = f;
            if (on_diag) a.dtab[(size_t)id * 4 + fa] = f;
            __threadfence();
        }
        __syncwarp();
        if (lane == 0) *((volatile int32_t *)(a.posid + pos)) = id;
    }
    if (id < 0) {
        if (lane == 0) a.status[2] = 1;
        return;
    }
    if (!won) {
        const double have = *((volatile const double *)(a.table + (size_t)id * 32 + lane));
        if (__ballot_sync(kFull, __double_as_longlong(have) != __double_as_longlong(f)) != 0u) {
            if (lane == 0) a.status[3] = 1;
            return;
        }
    }
    if (lane == 0) {
        if (u > 0 && a.diag_required && !isdiag) a.status[4] = 1;
        if (u == 0 && a.self_diag_required && !isdiag) a.status[5] = 1;  // the SD variants no longer apply: the plain ones take over
        a.ccode[slot] = id;
        if (a.dcode) {
            const int dir = u == 0 ? 0 : torus_direction(row, col, a.Lx, a.M);
            if (dir >= 0) a.dcode[(size_t)row * 5 + dir] = id;
        }
        if (a.dcode3) {
            const int dir = u == 0 ? 0 : cube_direction(row, col, a.Ly, a.Lz);
            if (dir >= 0) a.dcode3[(size_t)row * 8 + dir] = id;
        }
    }
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

// Build the block dictionary of the fixed-width matrix copy (e.idx / e.data must exist).
int dict_build(bdg_system *sys) {
    EllDev &e = sys->ell;
    e.dict_usable = false;
    e.n_unique = 0;
    const int64_t n_slots = e.n_sites * e.width;
    if (n_slots <= 0 || n_slots > (int64_t)1 << 30) return BDG_OK;
    // Worth it when the table is a small fraction of the matrix (each distinct block is still
    // read from HBM about once per step; the codes cost 4 bytes per slot).
    const int64_t max_unique = std::max<int64_t>(1, n_slots * env_int("BDG_DICT_MAX_PERCENT", 35) / 100);
    BDG_TRY(dev_alloc(sys, e.tmp_where, (size_t)n_slots * sizeof(int32_t)));
    BDG_TRY(ensure_scratch(sys, 2, 64));
    int *scal = sys->scratch_i32[2].as<int>();  // [0] keys inserted, [1] overflow, [2] distinct (scan), [3] mismatch
    const unsigned warps_grid = (unsigned)ceil_div(n_slots * 32, 256);
    // Lattice Hamiltonians have a handful of distinct blocks: start with a small table (cheap to
    // clear and to scan) and grow it only when it fills up.
    int64_t cap = 1 << 16;
    int host[4] = {0, 0, 0, 0};
    for (;;) {
        const int limit = (int)std::min<int64_t>(cap / 2, max_unique);
        BDG_TRY(dev_alloc(sys, e.tmp_keys, (size_t)cap * sizeof(unsigned long long)));
        BDG_TRY(dev_alloc(sys, e.tmp_rep, (size_t)cap * sizeof(int)));
        BDG_TRY(dev_alloc(sys, e.tmp_dense, (size_t)(n_slots + 1) * sizeof(int32_t)));
        BDG_CUDA(cudaMemsetAsync(e.tmp_keys.ptr, 0xff, (size_t)cap * sizeof(unsigned long long), sys->stream));
        BDG_CUDA(cudaMemsetAsync(e.tmp_rep.ptr, 0x7f, (size_t)cap * sizeof(int), sys->stream));
        BDG_CUDA(cudaMemsetAsync(scal, 0, 4 * sizeof(int), sys->stream));
        dict_insert<<<warps_grid, 256, 0, sys->stream>>>(n_slots, e.data.as<double>(), e.tmp_keys.as<unsigned long long>(),
                                                         e.tmp_rep.as<int>(), (unsigned)(cap - 1), e.tmp_where.as<int32_t>(),
                                                         scal, limit, scal + 1);
        BDG_CUDA(cudaGetLastError());
        BDG_CUDA(cudaMemcpyAsync(host, scal, 2 * sizeof(int), cudaMemcpyDeviceToHost, sys->stream));
        BDG_CUDA(cudaStreamSynchronize(sys->stream));
        e.n_unique = host[0];  // exact unless the pass was abandoned (then: at least this many)
        if (!host[1]) break;
        if (limit >= max_unique) return BDG_OK;  // too many distinct blocks: keep the plain format
        cap <<= 4;
    }
    dict_flag_reps<<<(unsigned)ceil_div(n_slots, 256), 256, 0, sys->stream>>>(n_slots, e.tmp_rep.as<int>(), e.tmp_where.as<int32_t>(),
                                                                              e.tmp_dense.as<int32_t>());
    BDG_CUDA(cudaGetLastError());
    BDG_TRY(exclusive_scan_i32(sys, e.tmp_dense.as<int32_t>(), e.tmp_dense.as<int32_t>(), n_slots, scal + 2));
    const int n_unique = host[0];
    // Head room for blocks that later scatters add (ell_patch): half as many again, at least 64 Ki, and never more than
    // three quarters of the hash table.
    e.hash_cap = cap;
    e.table_cap = std::min<int64_t>(std::max<int64_t>(n_unique + n_unique / 2, n_unique + 65536), cap * 3 / 4);
    e.table_cap = std::max<int64_t>(e.table_cap, n_unique);
    BDG_TRY(dev_alloc(sys, e.code, (size_t)n_slots * sizeof(int32_t)));
    BDG_TRY(dev_alloc(sys, e.table, (size_t)e.table_cap * 32 * sizeof(double)));
    BDG_TRY(dev_alloc(sys, e.posid, (size_t)cap * sizeof(int32_t)));
    BDG_TRY(dev_alloc(sys, e.counters, 8 * sizeof(int)));
    BDG_CUDA(cudaMemsetAsync(e.posid.ptr, 0xff, (size_t)cap * sizeof(int32_t), sys->stream));
    dict_emit<<<warps_grid, 256, 0, sys->stream>>>(n_slots, e.data.as<double>(), e.tmp_rep.as<int>(),
                                                   e.tmp_dense.as<int32_t>(), e.tmp_where.as<int32_t>(),
                                                   e.code.as<int32_t>(), e.table.as<double>(), n_unique, e.posid.as<int32_t>(),
                                                   scal + 3);
    BDG_CUDA(cudaGetLastError());
    BDG_CUDA(cudaMemcpyAsync(host + 2, scal + 2, 2 * sizeof(int), cudaMemcpyDeviceToHost, sys->stream));
    BDG_CUDA(cudaStreamSynchronize(sys->stream));
    e.dict_usable = host[3] == 0 && host[2] == n_unique;  // no hash collision, table fully written
    // Real-diagonal off-site blocks (DIAG kernels)?
    e.diag_usable = false;
    e.self_diag_usable = false;
    if (e.dict_usable) {
        BDG_TRY(dev_alloc(sys, e.dtab, (size_t)e.table_cap * 4 * sizeof(double)));
        BDG_TRY(dev_alloc(sys, e.tmp_rep, (size_t)std::max<int64_t>(cap, n_unique) * sizeof(int)));  // reuse as isdiag[]
        BDG_CUDA(cudaMemsetAsync(scal, 0, 2 * sizeof(int), sys->stream));
        dict_diag_table<<<(unsigned)ceil_div((int64_t)n_unique * 32, 256), 256, 0, sys->stream>>>(
            n_unique, e.table.as<double>(), e.dtab.as<double>(), e.tmp_rep.as<int>());
        dict_offsite_diag<<<(unsigned)ceil_div(n_slots, 256), 256, 0, sys->stream>>>(
            n_slots, e.width, e.code.as<int32_t>(), e.tmp_rep.as<int>(), scal);
        BDG_CUDA(cudaGetLastError());
        BDG_CUDA(cudaMemcpyAsync(host, scal, 2 * sizeof(int), cudaMemcpyDeviceToHost, sys->stream));
        BDG_CUDA(cudaStreamSynchronize(sys->stream));
        e.diag_usable = host[0] == 0;
        e.self_diag_usable = host[1] == 0;
    }
    return BDG_OK;
}

}  // namespace

void ell_release(bdg_system *sys) {
    dev_free(sys, sys->ell.idx);
    dev_free(sys, sys->ell.data);
    dev_free(sys, sys->ell.code);
    dev_free(sys, sys->ell.table);
    dev_free(sys, sys->ell.dtab);
    dev_free(sys, sys->ell.dcode);
    dev_free(sys, sys->ell.dcode3);
    dev_free(sys, sys->ell.tmp_keys);
    dev_free(sys, sys->ell.tmp_rep);
    dev_free(sys, sys->ell.tmp_where);
    dev_free(sys, sys->ell.tmp_dense);
    dev_free(sys, sys->ell.posid);
    dev_free(sys, sys->ell.counters);
    sys->ell = EllDev();
}

int ell_build(bdg_system *sys) {
    EllDev &e = sys->ell;
    if (e.valid) return BDG_OK;
    BDG_TRY(build_packed(sys));
    const BsrDev &m = sys->packed;
    const int n = (int)m.n_sites;
    e.usable = false;
    e.dict_usable = false;
    e.diag_usable = false;
    e.self_diag_usable = false;
    e.pair_usable = false;
    e.cube_usable = false;
    e.n_unique = 0;
    e.n_sites = n;
    if (n > 0) {
        BDG_TRY(ensure_scratch(sys, 2, 64));
        int *max_need = sys->scratch_i32[2].as<int>();
        BDG_CUDA(cudaMemsetAsync(max_need, 0, sizeof(int), sys->stream));
        ell_row_need<<<(unsigned)ceil_div(n, 256), 256, 0, sys->stream>>>(n, m.indptr.as<int32_t>(),
                                                                         m.indices.as<int32_t>(), max_need);
        BDG_CUDA(cudaGetLastError());
        int need = 0;
        BDG_CUDA(cudaMemcpyAsync(&need, max_need, sizeof(int), cudaMemcpyDeviceToHost, sys->stream));
        BDG_CUDA(cudaStreamSynchronize(sys->stream));
        const int width = std::max(need, 3);
        // Padding costs matrix traffic: accept it when small, or when the matrix is too small to matter.
        const bool cheap = (int64_t)n * width * 4 <= m.n_blocks * 5 || (int64_t)n * width <= (1 << 16);
        if (width <= 8 && cheap) {
            e.width = width;
            BDG_TRY(dev_alloc(sys, e.idx, (size_t)n * width * sizeof(int32_t)));
            BDG_TRY(dev_alloc(sys, e.data, (size_t)n * width * 32 * sizeof(double)));
            const int64_t threads = (int64_t)n * width * 32;
            ell_fill<<<(unsigned)ceil_div(threads, 256), 256, 0, sys->stream>>>(
                n, width, m.indptr.as<int32_t>(), m.indices.as<int32_t>(), m.data.as<double>(), e.idx.as<int32_t>(),
                e.data.as<double>());
            BDG_CUDA(cudaGetLastError());
            e.usable = true;
            BDG_TRY(dict_build(sys));
            BDG_TRY(pair_probe(sys));
            BDG_TRY(cube_probe(sys));
        }
    }
    e.valid = true;
    sys->stats[1] += 1;
    return BDG_OK;
}

int ell_patch(bdg_system *sys, int64_t n, const int32_t *klist, bool *ok) {
    EllDev &e = sys->ell;
    *ok = false;
    if (!sys->packed_valid || !e.valid || !sys->pack_flags.ptr || !sys->pack_pos.ptr) return BDG_OK;
    if (env_int("BDG_NO_PATCH", 0)) return BDG_OK;  // A/B: always rebuild
    if (n == 0) {
        *ok = true;
        return BDG_OK;
    }
    const bool dict = e.usable && e.dict_usable;
    if (e.usable && !dict && e.n_unique > 0) return BDG_OK;  // a dictionary was attempted and given up: rebuild decides again
    BDG_TRY(dev_alloc(sys, e.counters, 8 * sizeof(int)));
    int host[6] = {(int)e.n_unique, 0, 0, 0, 0, 0};
    BDG_CUDA(cudaMemcpyAsync(e.counters.ptr, host, sizeof(host), cudaMemcpyHostToDevice, sys->stream));
    PatchArgs a{};
    a.s_indices = sys->skel.indices.as<int32_t>();
    a.s_brow = sys->skel.brow.as<int32_t>();
    a.s_data = sys->skel.data.as<double>();
    a.flags = sys->pack_flags.as<int32_t>();
    a.pos = sys->pack_pos.as<int32_t>();
    a.p_data = sys->packed.data.as<double>();
    a.width = e.usable ? e.width : 0;
    a.cidx = e.idx.as<int32_t>();
    a.cdata = e.data.as<double>();
    a.ccode = e.code.as<int32_t>();
    a.dict = dict ? 1 : 0;
    a.keys = e.tmp_keys.as<unsigned long long>();
    a.posid = e.posid.as<int32_t>();
    a.cap_mask = (unsigned)(e.hash_cap - 1);
    a.table = e.table.as<double>();
    a.dtab = e.dtab.as<double>();
    a.table_cap = (int)e.table_cap;
    a.diag_required = e.diag_usable ? 1 : 0;
    a.self_diag_required = e.self_diag_usable && !e.diag_usable ? 1 : 0;  // (only the SD kernel relies on it)
    a.dcode = e.pair_usable ? e.dcode.as<int32_t>() : nullptr;
    a.Lx = sys->cubic[0];
    a.M = e.pair_M;
    a.dcode3 = e.cube_usable ? e.dcode3.as<int32_t>() : nullptr;
    a.Ly = sys->cubic[1];
    a.Lz = sys->cubic[2];
    a.status = e.counters.as<int>();
    patch_blocks<<<(unsigned)ceil_div(n * 32, 256), 256, 0, sys->stream>>>(n, klist, a);
    BDG_CUDA(cudaGetLastError());
    BDG_CUDA(cudaMemcpyAsync(host, e.counters.ptr, sizeof(host), cudaMemcpyDeviceToHost, sys->stream));
    BDG_CUDA(cudaStreamSynchronize(sys->stream));
    if (host[1] || host[2] || host[3] || host[4]) return BDG_OK;  // pattern / capacity / collision / DIAG precondition: rebuild
    e.n_unique = host[0];
    if (host[5]) e.self_diag_usable = false;  // an on-site block with off-diagonal entries: same format, MMA on-site product
    *ok = true;
    return BDG_OK;
}

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
