// Internal declarations shared by the libbdg translation units (not part of the ABI).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include <string>
#include <vector>

#include "bdg.h"

// ---- error plumbing ---------------------------------------------------------------------
void bdg_set_error(const char *fmt, ...);

#define BDG_CUDA(expr)                                                                      \
    do {                                                                                    \
        cudaError_t err__ = (expr);                                                         \
        if (err__ != cudaSuccess) {                                                         \
            bdg_set_error("%s failed at %s:%d: %s", #expr, __FILE__, __LINE__,             \
                          cudaGetErrorString(err__));                                       \
            return BDG_E_CUDA;                                                              \
        }                                                                                   \
    } while (0)

#define BDG_TRY(expr)                                                                       \
    do {                                                                                    \
        int rc__ = (expr);                                                                  \
        if (rc__ != BDG_OK) return rc__;                                                    \
    } while (0)

#define BDG_REQUIRE(cond, ...)                                                              \
    do {                                                                                    \
        if (!(cond)) {                                                                      \
            bdg_set_error(__VA_ARGS__);                                                     \
            return BDG_E_INVALID;                                                           \
        }                                                                                   \
    } while (0)

// First statement of every ABI function that takes a handle.
#define BDG_ENTER(sys)                                                                      \
    BDG_REQUIRE((sys) != nullptr, "null handle");                                           \
    BDG_CUDA(cudaSetDevice((sys)->device))

// ---- device buffers -----------------------------------------------------------------------
// Thin owner of one cudaMalloc'd array; tracks bytes per handle.
struct DevBuf {
    void *ptr = nullptr;
    size_t bytes = 0;
    template <class T> T *as() const { return static_cast<T *>(ptr); }
};

struct bdg_system;
int dev_alloc(bdg_system *sys, DevBuf &buf, size_t bytes);
void dev_free(bdg_system *sys, DevBuf &buf);

// ---- BSR structure on the device ---------------------------------------------------------
// data layout == scipy bsr_matrix.data: [nb][4][4] complex128 (re, im interleaved), 256 B/block.
struct BsrDev {
    int64_t n_sites = 0;
    int64_t n_blocks = 0;
    DevBuf indptr;   // int32 [n_sites + 1]
    DevBuf indices;  // int32 [n_blocks]   ascending within a row
    DevBuf brow;     // int32 [n_blocks]   block row of every block (skeleton only)
    DevBuf data;     // double2 [n_blocks * 16]
};

// Row traversal of the fixed-width step kernels (cheb_ell.cu).  The lattice is cut into work
// items = (patch of Pz x Py sites in the z-y plane, one site per warp of the CTA) x (segment of
// `seg_len` consecutive x); a CTA marches its patch along x, so the +-x neighbour records of a row
// are the records the same warp touched one and two steps earlier, and the +-y / +-z neighbours
// belong to the warps next to it: they are served by the SM's L1, not by L2.  Items are handed
// out segment-major (item = it * gridDim.x + blockIdx.x), so the grid still sweeps the lattice as
// one wavefront and every vector byte leaves HBM once.  Matrices without cubic geometry use the
// degenerate walk Lz = n_sites, Pz = warps per CTA, Lx = 1 (plain wavefront over consecutive rows).
struct RowWalk {
    int Lz = 1, Ly = 1, Lx = 1;  // extents (site = z + y*Lz + x*Ly*Lz)
    int Pz = 1, Py = 1;          // patch extents; Pz * Py = warps per CTA
    int nPz = 1, n_patches = 1;  // patches along z, patches in the plane
    int seg_len = 1, n_items = 1;
    int prefetch = 0;            // rows ahead (a multiple of Ly*Lz) whose records are prefetched into L1; 0 = off
};

// Work lists of the two-applications-per-pass kernels (device, ChebState::work_items; work_lists.h): CTA c works through
// pieces[cta_begin[c] .. cta_begin[c + 1]), a piece = (run, patch, x0, len).  A maximal sequence of pieces of one panel inside
// a CTA is a "run": its dot products go to partials[run]; run_panel[run] = its panel, and the runs of panel p are
// panel_runs[p] .. panel_runs[p + 1].  The classic plan has no lists (null pointers): n_ctas CTAs per panel, n_runs =
// n_ctas x panels.
struct WorkLists {
    const int4 *pieces = nullptr;
    const int *cta_begin = nullptr, *run_panel = nullptr, *panel_runs = nullptr;
    int n_ctas = 0, n_runs = 0;
};

// Item grid of the two-steps-per-pass kernel (cheb_pair.cu): x-planes of M sites, cut into patches of
// P owned sites; an item = (patch, segment of seg_len consecutive x), handed out segment-major.
struct PairWalk {
    int Lx = 1, M = 1;
    int open = 0;  // the plane has open ends (no in-plane wrap-around block): the rim patches own their rim site
    int P = 1, n_patches = 1;
    int seg_len = 1, n_segs = 1, n_items = 1;
    WorkLists lists;
};

// Item grid of the two-applications-per-pass kernel for three-dimensional lattices (cheb_cube.cu): the (y, z) plane
// is cut into nPy x nPz patches; an item = (patch, segment of seg_len consecutive x), handed out segment-major.
struct CubeWalk {
    int Lx = 1, Ly = 1, Lz = 1;
    int nPy = 1, nPz = 1, n_patches = 1;
    int seg_len = 1, n_segs = 1, n_items = 1;
    WorkLists lists;
};

// ---- Chebyshev state ----------------------------------------------------------------------
struct PlanSwitches;  // cheb_plan.h

// How the recursion advances (plan_stepping, cheb_plan.h); ChebState::kernel keeps the matrix format of the single-step kernel.
enum class Stepping {
    Single,     // one step per launch (cheb.cu, cheb_ell.cu)
    Pair,       // two steps per launch whenever two or more remain (cheb_pair.cu); T_1 and odd leftovers: single-step kernel
    EvenPlane,  // even-vector recursion E_{j+1} = 2 T_2(H~) E_j - E_{j-1} on one-dimensional x-planes (cheb_pair.cu)
    EvenCube,   // ... on a three-dimensional lattice (cheb_cube.cu, 4-column panels)
};

// Signatures of the recursion kernel families: BSR (cheb.cu), fixed-width / dictionary (cheb_ell.cu), two steps per pass on
// planes (cheb_pair.cu) and on three-dimensional lattices (cheb_cube.cu).
using StepKernel = void (*)(const int32_t *, const int32_t *, const double2 *, const double2 *, double2 *, int, double,
                            double, double *, unsigned *, double *, int);
using EllKernel = void (*)(const int32_t *, const int32_t *, const double *, const double *, const double2 *, double2 *,
                           int, int, double, double, int, int, double *, unsigned *, double *, const RowWalk);
using PairKernel = void (*)(const int32_t *, const double *, const double *, const double2 *, const double2 *, double2 *,
                            double2 *, int, int, double, double, double, int, double *, unsigned *, double *, const PairWalk);
using CubeKernel = void (*)(const int32_t *, const double *, const double *, const double2 *, double2 *, int, int, double,
                            double, double, int, double *, unsigned *, double *, const CubeWalk);

// A kernel the plan chose and its launch shape: set by the configure functions, launched as is.
template <class Kernel> struct Launch {
    Kernel fn = nullptr;
    dim3 grid;
    unsigned threads = 0;
    size_t smem = 0;
};

struct ChebState {
    bool active = false;
    int kernel = BDG_KERNEL_DMMA;
    int32_t n_cols = 0;       // user columns on this GPU
    int32_t panel_width = 8;  // PW: columns per panel (1, 2, 4 or 8)
    int32_t n_panels = 0;
    double scale = 1.0;
    int32_t steps_done = 0;   // recursion steps after T_1 (T_{steps_done+1} is current)
    int32_t dot_capacity = 0; // steps for which dot storage exists
    // Vectors: [panel][site][col_in_panel][alpha] complex128; cur = T_n, prev = T_{n-1}.
    // The pair kernel writes T_{n+1}, T_{n+2} into the two buffers that hold neither (vec[2], vec[3]
    // exist only then); the single-step kernels overwrite prev in place.
    DevBuf vec[4];
    int cur = 0, prev = 1;
    Stepping stepping = Stepping::Single;  // even-vector recursions: vec[cur] = T_n, vec[prev] = T_{n-2}
    bool even() const { return stepping == Stepping::EvenPlane || stepping == Stepping::EvenCube; }
    int t2_rows_normalized = 0;  // launches whose dot rows have been rewritten in the single-step format
    // What the plan launches (bdg_cheb_begin and the configure functions):
    Launch<StepKernel> bsr_first, bsr_next;  // DMMA / FMA: T_1 and every later step
    Launch<EllKernel> ell_step;              // ELL / DICT / DICT_DIAG: every single step
    Launch<PairKernel> two_step;             // Pair / EvenPlane
    Launch<CubeKernel> cube_step;            // EvenCube
    RowWalk walk;                            // ell_step's row traversal
    PairWalk pair_walk;
    CubeWalk cube_walk;
    bool onsite_per_row = false;  // two_step: on-site fragments fetched per row from the table (SELF) instead of held
    bool onsite_diag = false;     // two_step: real-diagonal on-site product (SD)
    int partial_runs = 0;         // the most partial-sum slots (runs) per panel any launch of the plan writes
    // dots[(step * 2 + which) * n_panels * PW + panel * PW + c]; which 0 = <T_n,T_n>, 1 = <T_{n+1},T_n>
    DevBuf dots;
    DevBuf partials;  // per-CTA partial dot products of the step in flight
    DevBuf tickets;   // uint32 [n_panels] arrival counters (last CTA reduces)
    DevBuf mu_tmp;    // staging for moment read-out
    DevBuf obs_tmp;   // staging for observables.cu (coefficients, energies, results)
    DevBuf work_items;  // work lists of a balanced plan (WorkLists)
    int64_t launches = 0;
    // Local accumulator (bdg_cheb_local_begin, observables.cu): every launch that writes T_n with n < local_coef.size()
    // adds local_coef[n] * T_n[4 site + alpha][col] to local_acc[read][alpha].  Cleared by bdg_cheb_begin.
    bool local = false;
    std::vector<double> local_coef;
    int64_t local_reads = 0;
    DevBuf local_off;  // int64 [n_reads]: element offset of (site, col, alpha = 0) in the panel layout
    DevBuf local_acc;  // double2 [n_reads][4]
    // Recursion kernels launched since bdg_cheb_begin (bdg_cheb_launched): distinct entry points in the order of their
    // first launch.  `last_launched` makes a launch of the same kernel as the one before cost one compare.
    std::vector<const void *> launched;
    const void *last_launched = nullptr;
};

static inline void note_launch(ChebState &st, const void *kernel) {
    if (kernel == st.last_launched) return;
    st.last_launched = kernel;
    for (const void *k : st.launched)
        if (k == kernel) return;
    st.launched.push_back(kernel);
}

// Direction codes (EllDev::dcode, dcode3): per site, the dictionary code of the row's block in each direction of a
// nearest-neighbour stencil, so that a kernel finds a row's blocks without any index.
constexpr int kPlaneCodes = 5;  // dcode (cheb_pair.cu): self, x-1, y-1, y+1, x+1 on the Lx x M torus
constexpr int kCubeCodes = 8;   // dcode3 (cheb_cube.cu): self, x-1, y-1, z-1, z+1, y+1, x+1, padding on the open lattice
constexpr int kNoBlock = -1;    // no block in that direction: the kernel multiplies by a zero fragment
constexpr int kNoSite = -2;     // dcode3 only: no lattice site in that direction of y / z: the kernel keeps what it holds
// The cube kernel holds its fragments in registers and takes a dictionary of at most this many distinct blocks.
constexpr int64_t kCubeMaxUnique = 64;

// Kernel-native copies of the packed matrix for the step kernels, built and patched by formats.cu.
// Fixed-width rows (cheb_ell.cu): every block row padded to `width` slots, slot 0 = the diagonal block (zero block if
// absent), then the other blocks in ascending column order; padding slots are zero blocks pointing at the row itself.
//   idx  int32  [n_sites][width]
//   data double [n_sites][width][4 (a)][2 (re, im)][4 (b)]   -- MMA B-fragment order, 256 B/block
struct EllDev {
    bool valid = false;
    bool usable = false;   // false: rows too long / too ragged, use the generic kernel
    int width = 0;
    int64_t n_sites = 0;
    DevBuf idx, data;
    // Block dictionary over the same slots (cheb_ell.cu, DICT kernels): the DISTINCT blocks of the
    // matrix, and one code per slot.  Usable when the distinct blocks are a small fraction of all.
    //   code  int32  [n_sites][width]          table double [n_unique][4][2][4]
    bool dict_usable = false;
    bool diag_usable = false;  // every block outside slot 0 is real and diagonal: dtab[n_unique][4] holds the diagonals
    bool self_diag_usable = false;  // every block IN slot 0 (on-site) is real and diagonal (cheb_step_ell<..., SD>)
    int64_t n_unique = 0;
    DevBuf code, table, dtab;
    // Two-steps-per-pass kernel (cheb_pair.cu): dictionary format + nearest-neighbour stencil on a
    // lattice whose x-planes are one-dimensional (pair_M sites per plane).
    bool pair_usable = false;
    bool pair_open = false;  // no block wraps around in-plane
    int pair_M = 0;
    DevBuf dcode;  // int32 [n_sites][kPlaneCodes]; kNoBlock = none
    // ... and its three-dimensional sibling (cheb_cube.cu): open nearest-neighbour stencil on a lattice with Ly, Lz >= 2,
    // real-diagonal hopping blocks, at most kCubeMaxUnique distinct blocks.
    bool cube_usable = false;
    DevBuf dcode3;  // int32 [n_sites][kCubeCodes]; kNoBlock = no block, kNoSite = no site in y / z
    DevBuf tmp_keys, tmp_rep, tmp_where, tmp_dense;  // hash-table scratch of the dictionary build (kept for rebuilds)
    // ... and what stays alive for incremental updates (ell_patch): the hash table itself (tmp_keys, `hash_cap` slots),
    // posid[hash position] = dictionary code (-1: unused), the table's capacity in entries, the device PatchStatus.
    DevBuf posid, counters;
    int64_t hash_cap = 0, table_cap = 0;
};

struct bdg_system {
    int device = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    int sm_count = 148;
    bool quiesced = false;     // being destroyed, stream drained: dev_free need not synchronise per buffer
    int64_t dev_bytes = 0;
    int cubic[3] = {0, 0, 0};  // (Lx, Ly, Lz) when built by bdg_create_cubic, else zeros

    BsrDev skel;           // full skeleton, values as scattered so far
    BsrDev packed;         // after eliminate_zeros (built lazily)
    bool packed_valid = false;
    DevBuf pack_flags;     // int32 [skel.n_blocks]: block kept in `packed` (non-zero)      } kept after the compaction so that a
    DevBuf pack_pos;       // int32 [skel.n_blocks]: its position there                      } later scatter can patch the copies
    // Hermiticity bookkeeping: the stored matrix passed max|M - M^H| <= herm_tol and every change since went through a
    // checked scatter -- then the next scatter only needs to look at the blocks it writes (and their transposes).
    bool herm_verified = false;
    double herm_tol = 0.0;
    int64_t stats[5] = {0, 0, 0, 0, 0};  // bdg_stats
    int packed_max_row = 0;  // longest block row of `packed` (picks the kernel's unroll)

    DevBuf scratch_i32[4];  // reusable scratch (counts, scans, flags, positions)
    DevBuf stage[10];       // uploaded entry lists: {i, j, values, k1, k2} x {hopping, pairing}
    DevBuf scalars;         // small device scalars (first_bad, max_dev, ...)
    void *host_scalars = nullptr;  // pinned mirror

    ChebState cheb;
    EllDev ell;
    DevBuf multi_send, multi_recv;  // moments of this GPU / of all GPUs around the NCCL collective (multi.cu)
};

// scan.cu
int exclusive_scan_i32(bdg_system *sys, const int32_t *in, int32_t *out, int64_t n,
                       int32_t *total_dev /* device, may be null */);

// assemble.cu
int build_packed(bdg_system *sys);
int ensure_scratch(bdg_system *sys, int which, size_t bytes);

// cheb.cu
void cheb_release(bdg_system *sys);     // free all Chebyshev buffers
void cheb_deactivate(bdg_system *sys);  // matrix changed: recursion state is stale, keep buffers
int t2_finish_dots(bdg_system *sys);    // T2 mode: dot rows -> single-step format (call before reading st.dots)

// observables.cu
// Local accumulator: add the terms of T_n (vector x_a) and T_{n+1} (x_b, may be null) that fall inside the series.
int local_accumulate(bdg_system *sys, int n, const void *x_a, const void *x_b);

// formats.cu
int ell_build(bdg_system *sys);                    // (re)build sys->ell from sys->packed when stale
// After a scatter: bring `packed` and the kernel-native copies (fixed-width rows, dictionary, direction codes) up to date
// for the `n` skeleton blocks listed in `klist` (device; < 0 = skip) instead of rebuilding them.  *ok = false: the zero
// pattern changed, the table is full, ...: the caller invalidates the copies and the next recursion rebuilds them.
int ell_patch(bdg_system *sys, int64_t n, const int32_t *klist, bool *ok);
void ell_release(bdg_system *sys);

// cheb_ell.cu
int ell_configure(bdg_system *sys, const PlanSwitches &sw);  // ChebState::ell_step and its row traversal
int ell_launch_step(bdg_system *sys, bool first, const void *x_cur, void *x_io, double *dots_step);

// cheb_pair.cu
int pair_configure(bdg_system *sys, const PlanSwitches &sw);  // ChebState::two_step and its patch / segment plan
int pair_launch(bdg_system *sys, const void *x_prev, const void *x_cur, void *x_next1, void *x_next2, double *dots_step);
int t2_launch(bdg_system *sys, bool first, const void *x_cur, void *x_io, double *dots_step);

// cheb_cube.cu
int cube_configure(bdg_system *sys, const PlanSwitches &sw);  // ChebState::cube_step: patch shape, segment plan
int cube_launch(bdg_system *sys, bool first, const void *x_cur, void *x_io, double *dots_step);

static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// Integer switch from the environment (INTEGRATION.md); unset or empty: `fallback`.
static inline int env_int(const char *name, int fallback) {
    const char *v = getenv(name);
    return v && *v ? atoi(v) : fallback;
}
