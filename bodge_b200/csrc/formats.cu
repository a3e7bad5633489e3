// The kernel-native copies of the packed matrix that the step kernels read (EllDev, bdg_internal.h): fixed-width block
// rows in MMA B-fragment order, the block dictionary with its real-diagonal tables, and the direction codes of the two
// stencil kernels.  ell_build makes them from `packed`; ell_patch keeps them current after a scatter that rewrites a few
// blocks.  What the format is -- fragment order, block key, real-diagonal test, stencil directions -- is written down
// once, at the top of this file, and both paths use it.
#include <algorithm>

#include "bdg_internal.h"
#include "cheb_device.cuh"

namespace {

// ---- the format ---------------------------------------------------------------------------------
// Fragment lane l of a stored block (cheb_ell.cu: B fragment, lane l = Bop[l % 4][l / 4]) holds part (re, im) of entry
// (a, b) of the 4x4 block, with a = l >> 3, part = (l >> 2) & 1, b = l & 3.  `src` is that double's position in skeleton
// order ([a][b][re, im], as `packed` and the skeleton store a block); `diag` is a when the lane holds the real part of a
// diagonal entry (a, a) -- its place in dtab[code][4] --, else -1.
struct FragLane {
    int src, diag;
};
__device__ __forceinline__ FragLane frag_lane(int l) {
    const int a = l >> 3, part = (l >> 2) & 1, b = l & 3;
    return {(a * 4 + b) * 2 + part, part == 0 && a == b ? a : -1};
}

// Warp-collective, lane l holding double l of a block in fragment order: the block is real and diagonal (every other real
// and imaginary part compares == 0).
__device__ __forceinline__ bool real_diagonal(double v, int lane) {
    return __ballot_sync(kFull, frag_lane(lane).diag < 0 && v != 0.0) == 0u;
}

// Distinct blocks are found with an open-addressing hash table keyed by a 64-bit hash of the block's 256 bytes; every
// slot is then compared bit for bit with its table entry, so a hash collision can only disable the format, never change
// a result.  The table outlives the build: ell_patch looks new blocks up in it with the same key.
constexpr unsigned long long kEmptyKey = ~0ull;

// Warp-collective, lane l holding double l of a block in fragment order: the block's key (never kEmptyKey).
__device__ __forceinline__ unsigned long long block_key(double v, int lane) {
    uint64_t h = mix64((uint64_t)__double_as_longlong(v) + 0x9E3779B97F4A7C15ull * (uint64_t)(lane + 1));
#pragma unroll
    for (int d = 16; d; d >>= 1) h += __shfl_xor_sync(kFull, h, d);
    h = mix64(h);
    return h == kEmptyKey ? 0x1234567ull : h;
}

// Stencil direction of block column `col` seen from `row` on the Lx x M torus, the index into a row of dcode: 0 = the row
// itself, 1 = x-1, 2 = y-1, 3 = y+1, 4 = x+1 (wrap-around included), -1 = none of these.  Lx, M >= 3 keep the five apart.
__device__ __forceinline__ int torus_direction(int row, int col, int Lx, int M) {
    const int xr = row / M, yr = row - xr * M, xc = col / M, yc = col - xc * M;
    int dx = xc - xr, dy = yc - yr;
    dx += dx < 0 ? Lx : 0;
    dy += dy < 0 ? M : 0;
    if (dx == 0) return dy == 0 ? 0 : (dy == M - 1 ? 2 : (dy == 1 ? 3 : -1));
    if (dy != 0) return -1;
    return dx == Lx - 1 ? 1 : (dx == 1 ? 4 : -1);
}

// Stencil direction of block column `col` seen from `row` on the OPEN Lx x Ly x Lz lattice (site = z + Lz (y + Ly x)), the
// index into a row of dcode3: 0 = the row itself, 1 = x-1, 2 = y-1, 3 = z-1, 4 = z+1, 5 = y+1, 6 = x+1, -1 = anything else
// (wrap-around included).
__device__ __forceinline__ int cube_direction(int row, int col, int Ly, int Lz) {
    const int zr = row % Lz, yr = (row / Lz) % Ly, xr = row / (Lz * Ly);
    const int zc = col % Lz, yc = (col / Lz) % Ly, xc = col / (Lz * Ly);
    const int dx = xc - xr, dy = yc - yr, dz = zc - zr;
    if (dy == 0 && dz == 0) return dx == 0 ? 0 : (dx == -1 ? 1 : (dx == 1 ? 6 : -1));
    if (dx == 0 && dz == 0) return dy == -1 ? 2 : (dy == 1 ? 5 : -1);
    if (dx == 0 && dy == 0) return dz == -1 ? 3 : (dz == 1 ? 4 : -1);
    return -1;
}

// ---- fixed-width rows -----------------------------------------------------------------------------
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

// One warp per (row, slot); lane l writes double l of the slot in fragment order.
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
    if (src >= 0) v = data[(size_t)(p0 + src) * 32 + frag_lane(lane).src];
    cdata[w * 32 + lane] = v;
    if (lane == 0) cidx[w] = src >= 0 ? indices[p0 + src] : row;
}

// ---- block dictionary -----------------------------------------------------------------------------
// One warp per slot: key, find-or-insert, remember the table position and the smallest slot id holding that key (the
// representative whose bytes become the table entry).  The table is sized for few distinct blocks; when more than `limit`
// keys have been inserted the pass is abandoned (*overflow = 1) and the host retries with a larger table or gives the
// format up.
__global__ void __launch_bounds__(256)
dict_insert(int64_t n_slots, const double *__restrict__ cdata, unsigned long long *__restrict__ keys,
            int *__restrict__ rep, unsigned cap_mask, int32_t *__restrict__ where, int *__restrict__ counter,
            int limit, int *__restrict__ overflow) {
    const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= n_slots) return;
    const unsigned long long h = block_key(cdata[w * 32 + lane], lane);
    if (lane != 0) return;
    unsigned pos = (unsigned)h & cap_mask;
    for (;;) {
        unsigned long long seen = *((volatile unsigned long long *)(keys + pos));  // cheap hit for repeated blocks
        if (seen == kEmptyKey) {
            seen = atomicCAS(keys + pos, kEmptyKey, h);
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

// dtab[code][a] = Re of diagonal entry (a, a) of table block `code`; isdiag[code] = the block is real and diagonal.
__global__ void __launch_bounds__(256)
dict_diag_table(int n_unique, const double *__restrict__ table, double *__restrict__ dtab, int *__restrict__ isdiag) {
    const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (w >= n_unique) return;
    const double v = table[(size_t)w * 32 + lane];
    const int a = frag_lane(lane).diag;
    const bool diag = real_diagonal(v, lane);
    if (a >= 0) dtab[(size_t)w * 4 + a] = v;
    if (lane == 0) isdiag[w] = diag;
}

// bad[0] = 1 if any slot other than slot 0 holds a block that is not real-diagonal, bad[1] = 1 if any slot 0 does.
__global__ void __launch_bounds__(256)
dict_offsite_diag(int64_t n_slots, int width, const int32_t *__restrict__ ccode, const int *__restrict__ isdiag,
                  int *__restrict__ bad) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_slots) return;
    if (!isdiag[ccode[t]]) bad[t % width == 0 ? 1 : 0] = 1;
}

// ---- direction codes -----------------------------------------------------------------------------
// dcode[row]: the row's dictionary codes in the plane stencil's directions (bdg_internal.h: kPlaneCodes).  Slot 0 of the
// fixed-width copy is the diagonal block; padding slots point at the row itself.  flags[0] = 1 if some block column is
// none of the five on the (x, in-plane) torus -- the open stencil and the reference's periodic one both qualify --,
// flags[1] = 1 if some block wraps around in-plane.
__global__ void __launch_bounds__(256)
pair_codes(int n_sites, int width, int Lx, int M, const int32_t *__restrict__ cidx, const int32_t *__restrict__ ccode,
           int32_t *__restrict__ dcode, int *__restrict__ flags) {
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n_sites) return;
    const int y = row % M;
    int out[kPlaneCodes] = {kNoBlock, kNoBlock, kNoBlock, kNoBlock, kNoBlock};
    out[0] = ccode[(size_t)row * width];
    for (int u = 1; u < width; ++u) {
        const int d = torus_direction(row, cidx[(size_t)row * width + u], Lx, M);
        if (d < 0) flags[0] = 1;
        else if (d > 0) out[d] = ccode[(size_t)row * width + u];
    }
#pragma unroll
    for (int k = 0; k < kPlaneCodes; ++k) dcode[(size_t)row * kPlaneCodes + k] = out[k];
    if ((y == 0 && out[2] >= 0) || (y == M - 1 && out[3] >= 0)) flags[1] = 1;
}

// dcode3[row]: the row's dictionary codes in the cube stencil's directions (bdg_internal.h: kCubeCodes), kNoSite where the
// open lattice has no site in y / z.  *bad = 1 if some block column is none of the seven (padding slots point at the row
// itself).
__global__ void __launch_bounds__(256)
cube_codes(int n_sites, int width, int Ly, int Lz, const int32_t *__restrict__ cidx, const int32_t *__restrict__ ccode,
           int32_t *__restrict__ dcode, int *__restrict__ bad) {
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n_sites) return;
    const int z = row % Lz, y = (row / Lz) % Ly;
    int out[kCubeCodes] = {kNoBlock, kNoBlock, kNoBlock, kNoBlock, kNoBlock, kNoBlock, kNoBlock, kNoBlock};
    if (y == 0) out[2] = kNoSite;
    if (z == 0) out[3] = kNoSite;
    if (z == Lz - 1) out[4] = kNoSite;
    if (y == Ly - 1) out[5] = kNoSite;
    for (int u = 0; u < width; ++u) {
        const int col = cidx[(size_t)row * width + u];
        if (u > 0 && col == row) continue;  // padding
        const int d = u == 0 ? 0 : cube_direction(row, col, Ly, Lz);
        if (d >= 0) out[d] = ccode[(size_t)row * width + u];
        else *bad = 1;
    }
#pragma unroll
    for (int k = 0; k < kCubeCodes; ++k) dcode[(size_t)row * kCubeCodes + k] = out[k];
}

// ---- incremental update after a scatter (SURVEY 8f-3: re-enter `with`, change a few terms, ask again) -----------
// One warp per touched skeleton block: copy it into its place in `packed`, into its fixed-width slot (fragment order), look
// it up in -- or add it to -- the dictionary and rewrite the slot's code (and direction code).
struct PatchStatus {
    int n_unique;          // distinct blocks so far: a new block takes this code
    int pattern_changed;   // a block became zero or non-zero
    int table_full;
    int hash_collision;
    int offsite_not_diag;  // an off-site block that is not real-diagonal: the DIAG kernels no longer apply
    int onsite_not_diag;   // an on-site block that is not: the SD kernels no longer apply
};
constexpr size_t kCounterBytes = 8 * sizeof(int);  // EllDev::counters
static_assert(sizeof(PatchStatus) <= kCounterBytes, "EllDev::counters holds a PatchStatus");

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
    PatchStatus *status;
};

__global__ void __launch_bounds__(256)
patch_blocks(int64_t n, const int32_t *__restrict__ klist, const PatchArgs a) {
    const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= n) return;
    const int k = klist[w];
    if (k < 0) return;
    const double vs = a.s_data[(size_t)k * 32 + lane];  // skeleton order
    const bool nz = __ballot_sync(kFull, vs != 0.0) != 0u;
    if (nz != (a.flags[k] != 0)) {
        if (lane == 0) a.status->pattern_changed = 1;
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
            if (lane == 0) a.status->pattern_changed = 1;
            return;
        }
        u = __ffs(m) - 1;
    }
    const int64_t slot = (int64_t)row * a.width + u;
    const FragLane fl = frag_lane(lane);
    const double f = a.s_data[(size_t)k * 32 + fl.src];
    a.cdata[slot * 32 + lane] = f;
    if (!a.dict) return;
    const unsigned long long h = block_key(f, lane);
    int id = -1, won = 0;
    unsigned pos = 0;
    if (lane == 0) {
        pos = (unsigned)h & a.cap_mask;
        for (;;) {
            unsigned long long seen = *((volatile unsigned long long *)(a.keys + pos));
            if (seen == kEmptyKey) {
                seen = atomicCAS(a.keys + pos, kEmptyKey, h);
                if (seen == kEmptyKey) {
                    won = 1;
                    id = atomicAdd(&a.status->n_unique, 1);
                    if (id >= a.table_cap) {
                        a.status->table_full = 1;
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
    const bool isdiag = real_diagonal(f, lane);
    if (won) {
        if (id >= 0) {
            a.table[(size_t)id * 32 + lane] = f;
            if (fl.diag >= 0) a.dtab[(size_t)id * 4 + fl.diag] = f;
            __threadfence();
        }
        __syncwarp();
        if (lane == 0) *((volatile int32_t *)(a.posid + pos)) = id;
    }
    if (id < 0) {
        if (lane == 0) a.status->table_full = 1;
        return;
    }
    if (!won) {
        const double have = *((volatile const double *)(a.table + (size_t)id * 32 + lane));
        if (__ballot_sync(kFull, __double_as_longlong(have) != __double_as_longlong(f)) != 0u) {
            if (lane == 0) a.status->hash_collision = 1;
            return;
        }
    }
    if (lane == 0) {
        if (u > 0 && a.diag_required && !isdiag) a.status->offsite_not_diag = 1;
        if (u == 0 && a.self_diag_required && !isdiag) a.status->onsite_not_diag = 1;
        a.ccode[slot] = id;
        if (a.dcode) {
            const int dir = u == 0 ? 0 : torus_direction(row, col, a.Lx, a.M);
            if (dir >= 0) a.dcode[(size_t)row * kPlaneCodes + dir] = id;
        }
        if (a.dcode3) {
            const int dir = u == 0 ? 0 : cube_direction(row, col, a.Ly, a.Lz);
            if (dir >= 0) a.dcode3[(size_t)row * kCubeCodes + dir] = id;
        }
    }
}

// ---- host side ------------------------------------------------------------------------------------
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
    BDG_TRY(dev_alloc(sys, e.counters, kCounterBytes));
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

// Direction codes of the two-steps-per-pass kernel (cheb_pair.cu) when the copy qualifies: dictionary built,
// one-dimensional x-planes of >= 3 sites, >= 3 planes, rows of <= 5 blocks, nearest-neighbour stencil (open or periodic).
int pair_probe(bdg_system *sys) {
    EllDev &e = sys->ell;
    e.pair_usable = false;
    e.pair_M = 0;
    if (!e.usable || !e.dict_usable || e.width > 5 || e.width < 3) return BDG_OK;
    const int Lx = sys->cubic[0], Ly = sys->cubic[1], Lz = sys->cubic[2];
    if ((int64_t)Lx * Ly * Lz != e.n_sites) return BDG_OK;
    const int M = Lz == 1 ? Ly : (Ly == 1 ? Lz : 0);
    if (M < 3 || Lx < 3) return BDG_OK;
    BDG_TRY(ensure_scratch(sys, 2, 64));
    int *flags = sys->scratch_i32[2].as<int>();  // pair_codes: [0] outside the stencil, [1] wraps around in-plane
    BDG_CUDA(cudaMemsetAsync(flags, 0, 2 * sizeof(int), sys->stream));
    BDG_TRY(dev_alloc(sys, e.dcode, (size_t)e.n_sites * kPlaneCodes * sizeof(int32_t)));
    pair_codes<<<(unsigned)ceil_div(e.n_sites, 256), 256, 0, sys->stream>>>((int)e.n_sites, e.width, Lx, M, e.idx.as<int32_t>(),
                                                                          e.code.as<int32_t>(), e.dcode.as<int32_t>(), flags);
    BDG_CUDA(cudaGetLastError());
    int host[2] = {1, 1};
    BDG_CUDA(cudaMemcpyAsync(host, flags, sizeof(host), cudaMemcpyDeviceToHost, sys->stream));
    BDG_CUDA(cudaStreamSynchronize(sys->stream));
    e.pair_M = M;
    if (host[0]) {
        dev_free(sys, e.dcode);
        return BDG_OK;
    }
    e.pair_usable = true;
    // Open plane ends let the rim patches own their rim site; the flag stays valid under incremental updates, which cannot
    // add a block (a changed zero pattern rebuilds everything).
    e.pair_open = host[1] == 0;
    return BDG_OK;
}

// Direction codes of the even-vector kernel for three-dimensional lattices (cheb_cube.cu) when the copy qualifies:
// dictionary with real-diagonal hopping blocks and at most kCubeMaxUnique entries, cubic lattice with Lx, Ly, Lz >= 2,
// open nearest-neighbour stencil.
int cube_probe(bdg_system *sys) {
    EllDev &e = sys->ell;
    e.cube_usable = false;
    if (!e.usable || !e.dict_usable || !e.diag_usable || e.width > 7 || e.n_unique > kCubeMaxUnique) return BDG_OK;
    const int Lx = sys->cubic[0], Ly = sys->cubic[1], Lz = sys->cubic[2];
    if ((int64_t)Lx * Ly * Lz != e.n_sites || Lx < 2 || Ly < 2 || Lz < 2) return BDG_OK;
    if (e.n_sites * kCubeCodes > (int64_t)1 << 30) return BDG_OK;
    BDG_TRY(ensure_scratch(sys, 2, 64));
    int *bad = sys->scratch_i32[2].as<int>();
    BDG_CUDA(cudaMemsetAsync(bad, 0, sizeof(int), sys->stream));
    BDG_TRY(dev_alloc(sys, e.dcode3, (size_t)e.n_sites * kCubeCodes * sizeof(int32_t)));
    cube_codes<<<(unsigned)ceil_div(e.n_sites, 256), 256, 0, sys->stream>>>((int)e.n_sites, e.width, Ly, Lz, e.idx.as<int32_t>(),
                                                                          e.code.as<int32_t>(), e.dcode3.as<int32_t>(), bad);
    BDG_CUDA(cudaGetLastError());
    int host = 1;
    BDG_CUDA(cudaMemcpyAsync(&host, bad, sizeof(int), cudaMemcpyDeviceToHost, sys->stream));
    BDG_CUDA(cudaStreamSynchronize(sys->stream));
    if (host != 0) {
        dev_free(sys, e.dcode3);
        return BDG_OK;
    }
    e.cube_usable = true;
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
    BDG_TRY(dev_alloc(sys, e.counters, kCounterBytes));
    PatchStatus status{};
    status.n_unique = (int)e.n_unique;
    BDG_CUDA(cudaMemcpyAsync(e.counters.ptr, &status, sizeof(status), cudaMemcpyHostToDevice, sys->stream));
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
    // The single-step SD kernel (ell_configure) is picked whenever self_diag_usable holds, real-diagonal hopping or not: a
    // forced "dict" runs it on a matrix that also qualifies for "dict_diag".
    a.self_diag_required = e.self_diag_usable ? 1 : 0;
    a.dcode = e.pair_usable ? e.dcode.as<int32_t>() : nullptr;
    a.Lx = sys->cubic[0];
    a.M = e.pair_M;
    a.dcode3 = e.cube_usable ? e.dcode3.as<int32_t>() : nullptr;
    a.Ly = sys->cubic[1];
    a.Lz = sys->cubic[2];
    a.status = e.counters.as<PatchStatus>();
    patch_blocks<<<(unsigned)ceil_div(n * 32, 256), 256, 0, sys->stream>>>(n, klist, a);
    BDG_CUDA(cudaGetLastError());
    BDG_CUDA(cudaMemcpyAsync(&status, e.counters.ptr, sizeof(status), cudaMemcpyDeviceToHost, sys->stream));
    BDG_CUDA(cudaStreamSynchronize(sys->stream));
    if (status.pattern_changed || status.table_full || status.hash_collision || status.offsite_not_diag) return BDG_OK;  // rebuild
    e.n_unique = status.n_unique;
    // The copies stay; what no longer holds takes its kernels out of the plan until the next rebuild.
    if (status.onsite_not_diag) e.self_diag_usable = false;  // an on-site block with off-diagonal entries: MMA on-site product
    if (e.n_unique > kCubeMaxUnique) e.cube_usable = false;   // more distinct blocks than the cube kernel holds in registers
    *ok = true;
    return BDG_OK;
}
