/*
 * bdg.h -- C ABI of libbdg: B200-native (sm_100a) BdG Hamiltonian assembly and
 * Chebyshev/KPM expansion.  This is the drop-in boundary for the numerical hot path of
 * jabirali/bodge v1.3.0; every entry point names the reference code it replaces
 * (paths relative to the reference checkout).
 *
 * Conventions
 *   - plain C types only; all arrays are caller-owned and borrowed for the duration of a call;
 *   - host pointers unless a parameter says "device";
 *   - every function returns 0 on success or a BDG_E_* code; bdg_last_error() gives the text
 *     of the last failure on the calling thread;
 *   - one bdg_t owns all device memory of one Hamiltonian on one GPU and one CUDA stream
 *     (its own by default, or a borrowed one via bdg_set_stream); not thread-safe per handle;
 *   - complex numbers are interleaved (re, im) doubles = numpy complex128;
 *   - site indices are the lattice's flat indices (bodge/lattice.py:101-108), scalar rows are
 *     4*site + alpha with alpha in (e-up, e-down, h-up, h-down) (bodge README.md:110-115).
 */
#ifndef BDG_H
#define BDG_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BDG_ABI_VERSION 1

enum {
    BDG_OK = 0,
    BDG_E_INVALID = 1,       /* bad argument / bad state            -> ValueError / RuntimeError      */
    BDG_E_CUDA = 2,          /* CUDA runtime failure                -> RuntimeError                   */
    BDG_E_NOT_NEIGHBOUR = 3, /* (i,j) is not a block of the skeleton -> IndexError  (hamiltonian.py:170) */
    BDG_E_NOT_HERMITIAN = 4, /* max|M - M^H| > tol                  -> RuntimeError (hamiltonian.py:122) */
    BDG_E_OUT_OF_BOUNDS = 5, /* site index outside [0, N)           -> ValueError   (lattice.py:106)  */
    BDG_E_NO_DEVICE = 6      /* no usable CUDA device               -> RuntimeError                   */
};

typedef struct bdg_system bdg_t;

/* ---- housekeeping ------------------------------------------------------------------ */
int bdg_abi_version(void);
const char *bdg_last_error(void);
int bdg_device_count(int *count);
int bdg_destroy(bdg_t *sys);
/* Device buffers released by a handle are kept in a per-device cache and handed to the next
 * handle that asks for that size (cudaMalloc / cudaFree of a 1.3 GB block array cost milliseconds; the
 * reference has no counterpart -- numpy's allocator plays this role for its `_matrix.data`).  At most
 * BDG_CACHE_MB (default 8192, 0 = off) are held; this returns them to the driver. */
int bdg_release_cached(int device);
/* Borrow a CUDA stream (cudaStream_t / CUstream as void*); NULL restores the handle's own. */
int bdg_set_stream(bdg_t *sys, void *stream);
int bdg_sync(bdg_t *sys);
/* Bytes of device memory currently owned by the handle. */
int bdg_device_bytes(bdg_t *sys, int64_t *bytes);
/* Page-locked host buffers for callers that want full-rate host<->device copies of the packed
 * entry arrays (any host memory works; pageable memory is staged by the driver). */
int bdg_pinned_alloc(int64_t bytes, void **out);
int bdg_pinned_free(void *ptr);

/* ---- skeleton: replaces Hamiltonian.__init__ (bodge/hamiltonian.py:25-67) ------------ */
/* Periodic-stencil skeleton of CubicLattice((Lx,Ly,Lz)) built on the device: per-site sorted,
 * de-duplicated neighbour lists in registers, warp-shuffle scan for indptr.  Equals what the
 * reference obtains from lattice.sites() + bonds() + edges() through scipy coo->bsr. */
int bdg_create_cubic(int device, int32_t Lx, int32_t Ly, int32_t Lz, bdg_t **out);
/* Any Lattice subclass: pairs (i,j) as yielded by `for ri, rj in lattice` (flat indices).
 * Both orientations are inserted, duplicates merged, rows sorted (bucket-by-row + per-row sort). */
int bdg_create_generic(int device, int64_t n_sites, int64_t n_pairs, const int32_t *pair_i,
                       const int32_t *pair_j, bdg_t **out);
int bdg_skeleton_sizes(bdg_t *sys, int64_t *n_sites, int64_t *n_blocks);

/* ---- block lookup: replaces Hamiltonian.index (bodge/hamiltonian.py:157-170) --------- */
/* k[e] = position of block (i[e], j[e]) in the skeleton's data array.  BDG_E_NOT_NEIGHBOUR /
 * BDG_E_OUT_OF_BOUNDS with *bad_entry = first offending e otherwise. */
int bdg_lookup(bdg_t *sys, int64_t n, const int32_t *i, const int32_t *j, int64_t *k,
               int64_t *bad_entry);

/* ---- scatter: replaces Hamiltonian.__exit__ (bodge/hamiltonian.py:91-126) ------------ */
/* h_val / p_val: [n,2,2] complex128.  For every hopping entry  blk(i,j)[0:2,0:2] = H,
 * blk(i,j)[2:4,2:4] = -conj(H); for every pairing entry  blk(i,j)[0:2,2:4] = D,
 * blk(j,i)[2:4,0:2] = D^dagger.  Keys must be unique within each list (they come from a dict).
 * As in the reference, entries before the first failing lookup are applied and the rest are not
 * (hopping entries first, then pairing), and the Hermitian check runs last:
 * *max_dev = max|M - M^H|; returns BDG_E_NOT_HERMITIAN when it exceeds herm_tol (state stays
 * modified, like the reference).  herm_tol < 0 skips the check. */
int bdg_scatter(bdg_t *sys, int64_t n_hop, const int32_t *h_i, const int32_t *h_j,
                const double *h_val, int64_t n_pair, const int32_t *p_i, const int32_t *p_j,
                const double *p_val, double herm_tol, double *max_dev, int64_t *bad_entry);
/* Set every stored value back to zero (fresh skeleton). */
int bdg_clear(bdg_t *sys);
/* Incremental updates (the reference's parameter-sweep idiom: re-enter `with` for a few keys, ask for an observable
 * again -- tests/test_physics.py:155-160, 221-224; its scatter touches only the keys set, bodge/hamiltonian.py:102-118).
 * bdg_scatter patches the compacted matrix and the step kernels' own copies of it (fixed-width rows, block dictionary,
 * direction codes) for the blocks it writes, and checks Hermiticity on those blocks only, whenever it rewrites at most a
 * quarter of the blocks, the zero pattern is unchanged and the stored matrix had passed the check before; otherwise the
 * copies are rebuilt by the next recursion.
 * out[0] = compactions (eliminate_zeros) so far, out[1] = builds of the kernel-native copies, out[2] = scatters that
 * were patched in place, out[3] = blocks patched, out[4] = Hermitian checks restricted to the written blocks. */
int bdg_stats(bdg_t *sys, int64_t out[5]);

/* ---- export: replaces Hamiltonian.matrix("bsr") / ._matrix (bodge/hamiltonian.py:128-143) */
/* Two-phase: call with indptr = indices = data = NULL to get *n_blocks, then with buffers
 * indptr[N+1] int32, indices[nb] int32, data[nb*32] double.  eliminate_zeros != 0 drops every
 * block whose 16 entries all compare == 0 (scipy bsr eliminate_zeros), else the full skeleton. */
int bdg_export_bsr(bdg_t *sys, int eliminate_zeros, int64_t *n_blocks, int32_t *indptr,
                   int32_t *indices, double *data);
/* Scalar-level exports of the 4N x 4N matrix: replace matrix("csr") / matrix("csc") / matrix("dense")
 * (bodge/hamiltonian.py:144-151: scipy tocsr()/tocsc() + eliminate_zeros(), todense()).
 * bdg_export_csr: transpose = 0 gives CSR, 1 gives CSC; int32 indptr[4N+1] and indices[nnz] (ascending
 * inside every row / column), data[nnz] complex128; explicit zeros are dropped.  Two-phase like
 * bdg_export_bsr: indices = data = NULL returns *nnz (and indptr if given).
 * bdg_export_dense: out[4N][4N] complex128, row-major. */
int bdg_export_csr(bdg_t *sys, int transpose, int64_t *nnz, int32_t *indptr, int32_t *indices, double *data);
int bdg_export_dense(bdg_t *sys, double *out);
/* out[e] = the stored block at skeleton position k[e] (from bdg_lookup), [4][4] complex128 row-major: n * 32 doubles.
 * A few chosen blocks without exporting the matrix, e.g. the periodic-edge blocks of one lattice axis, to learn whether
 * any of them is non-zero (whether that axis wraps).  BDG_E_INVALID names the first position outside the skeleton. */
int bdg_gather_blocks(bdg_t *sys, int64_t n, const int64_t *k, double *out);
/* Overwrite all stored values from a host array laid out like the skeleton's data (inverse of
 * export with eliminate_zeros = 0; used for `system._data[...] = ...` style direct edits). */
int bdg_import_data(bdg_t *sys, const double *data);

/* ---- spectral bound -------------------------------------------------------------------- */
/* *norm = max absolute row sum of the 4N x 4N matrix (>= spectral radius). */
int bdg_norm_inf(bdg_t *sys, double *norm);

/* ---- Chebyshev / KPM engine (no reference code; arithmetic = scipy bsr_matvecs on
 *      matrix("bsr"), consumers = free_energy / ldos, bodge/hamiltonian.py:253-387) --------- */
enum { BDG_X0_PROBE = 0, BDG_X0_RADEMACHER = 1, BDG_X0_CLASS = 2 };
enum { BDG_MU_PER_COLUMN = 0, BDG_MU_SUM = 1 };
/* AUTO = PAIR where it applies (DICT / DICT_DIAG matrix, nearest-neighbour stencil on a lattice with one-dimensional
 *        x-planes, >= 5 columns), else DICT_DIAG, else DICT, else ELL -- the first the matrix qualifies for -- else DMMA.
 *        BDG_AUTO_PAIR=0 in the environment keeps AUTO / AUTO_MOMENTS on the single-step kernels.
 * AUTO_MOMENTS = AUTO for callers that only read moments / observables (never T_{n-1}): T2 where PAIR would be
 *        chosen, else as AUTO.  bdg_cheb_moments and the Python observables use it;
 * T2   = the even-vector ("doubled argument") recursion E_{j+1} = 2 T_2(H~) E_j - E_{j-1}, E_j = T_2j(H~) x, on the
 *        PAIR kernel: two applications of H~ per launch like PAIR, but only T_n and T_{n-2} are kept, so a launch
 *        moves three vector passes instead of four and two buffers suffice.  The four dot products of a launch
 *        (<E_j,E_j>, <H~E_j,E_j>, <E_{j+1},E_j>, <E_{j+1},H~E_j>) give the same four moments through
 *        T_m T_n = (T_{m+n} + T_|m-n|)/2 (odd ones by a two-term recurrence).  Steps advance in twos (an odd
 *        bdg_cheb_steps request is rounded up), bdg_cheb_begin already performs the first (T_2), and
 *        bdg_cheb_vectors(which = 1) is not available.  Same requirements as PAIR (open or periodic stencil) -- or a
 *        THREE-DIMENSIONAL lattice (Ly, Lz >= 2) with an open nearest-neighbour stencil, real-diagonal hopping blocks,
 *        <= 64 distinct blocks and >= 3 columns: there it runs on 4-column panels (bdg_cheb_info: panel_width = 4) with a
 *        kernel of its own (csrc/cheb_cube.cu), which AUTO_MOMENTS prefers when its work items fill the GPU (e.g. 64^3 sites
 *        with >= 8 columns); BDG_AUTO_CUBE=0 in the environment switches that preference off;
 * PAIR = two recursion steps per launch on the DICT / DICT_DIAG format: T_{n+1} is consumed out of shared
 *        memory instead of coming back from HBM, so two steps move four vector passes instead of six.  Needs
 *        >= 5 columns and a lattice with one-dimensional x-planes (Lz = 1 or Ly = 1) whose stored blocks form
 *        an open nearest-neighbour stencil; vectors bit-identical to DICT / DICT_DIAG.  T_1 and an odd
 *        leftover step run on the single-step kernel of the same format;
 * DICT_DIAG = DICT for matrices whose blocks off the lattice diagonal are all real and diagonal (hopping
 *        -t sigma_0 / m sigma_3 without pairing on the bonds): those blocks cost two DFMA instead of two
 *        FP64 MMAs.  Same sums in a different rounding order than DICT / ELL (agrees to ~1e-15);
 * DICT = the ELL kernel on a block-dictionary copy of the matrix: the distinct 4x4 blocks once, plus a
 *        4-byte code per block.  Lattice Hamiltonians repeat a handful of hopping / on-site blocks
 *        millions of times, so the per-step matrix traffic drops from 260 to 8 bytes per block; the
 *        arithmetic and its order are those of ELL (vectors bit-identical; moments too when the grids agree).  Chosen when the
 *        distinct blocks are <= 35 % of all blocks;
 * ELL  = FP64 warp-MMA on the kernel-native fixed-width row format (block rows of <= 8 blocks: every
 *        lattice Hamiltonian), one pass over the matrix serving up to 32 columns;
 * DMMA = FP64 warp-MMA on the BSR arrays as exported (any row length);
 * FMA  = scalar formulation (A/B reference).
 * 4 and 5 are unassigned: bdg_cheb_begin refuses them, and they are not to be reused, so that a caller built against an
 * older header gets an error instead of another kernel. */
enum { BDG_KERNEL_AUTO = 0, BDG_KERNEL_DMMA = 1, BDG_KERNEL_FMA = 2, BDG_KERNEL_ELL = 3,
       BDG_KERNEL_DICT = 6, BDG_KERNEL_DICT_DIAG = 7,
       BDG_KERNEL_PAIR = 8, BDG_KERNEL_T2 = 9, BDG_KERNEL_AUTO_MOMENTS = 10 };

/* Distance classes of the sites for BDG_X0_CLASS start vectors: site_class[i] in [0, n_classes) for every site i < n_sites
 * (n_sites must be the skeleton's).  Uploaded once and kept by the handle for every later recursion until the next call;
 * BDG_E_INVALID names the first bad entry.  The caller chooses the classes so that two distinct sites of one class are
 * far apart in the graph of the stored blocks: a polynomial p(H~) of degree m has no element between sites more than m
 * hops apart, so a class column read at one of its sites gives p(H~)'s element there plus those to the class's other
 * sites (Hamiltonian.density_matrix(spacing=...)). */
int bdg_set_classes(bdg_t *sys, int64_t n_sites, const int32_t *site_class, int32_t n_classes);

/* Start a recursion on n_cols start vectors resident on this GPU.
 *   kind = BDG_X0_PROBE:      column c = unit vector e_{probe_rows[c]}           (LDOS-type)
 *   kind = BDG_X0_RADEMACHER: column c = +-1 vector hashed from (seed, row, col_offset + c)
 *   kind = BDG_X0_CLASS:      column c = sum of e_{4i+beta} over the sites i of class k (bdg_set_classes), given as the
 *                             "class row" probe_rows[c] = 4k + beta, beta in 0..3 -- the probe row of a class instead
 *                             of a site; k >= n_classes is refused with the column named
 * scale = a  (H~ = H / a must have its spectrum inside [-1, 1]).
 * Builds T_0 = X0 and T_1 = H~ T_0 and the first two dot products. */
int bdg_cheb_begin(bdg_t *sys, int kind, int32_t n_cols, const int64_t *probe_rows, uint64_t seed,
                   int64_t col_offset, double scale, int kernel);
/* Enqueue n_steps fused steps T_{n+1} = 2 H~ T_n - T_{n-1} (+ <T_n,T_n>, <T_{n+1},T_n>).
 * elapsed_ms != NULL: bracket the steps with CUDA events on the handle's stream, synchronise,
 * and return the device time. */
int bdg_cheb_steps(bdg_t *sys, int32_t n_steps, float *elapsed_ms);
/* Pre-size the dot-product storage for n_steps further steps (bdg_cheb_steps grows it on demand,
 * which costs an allocation and a stream synchronisation the first time). */
int bdg_cheb_reserve(bdg_t *sys, int32_t n_steps);
/* Moments available so far: 2 * (steps + 1). */
int bdg_cheb_available(bdg_t *sys, int32_t *n_moments);
/* mu[n * n_out + c], n < n_moments; n_out = n_cols (BDG_MU_PER_COLUMN) or 1 (BDG_MU_SUM, summed
 * over this GPU's columns).  mu_on_device != 0: mu is a device pointer (e.g. for an NCCL reduce). */
int bdg_cheb_moments_read(bdg_t *sys, int32_t n_moments, int reduce, double *mu, int mu_on_device);
/* Convenience: begin + ceil(n_moments/2)-1 steps + read. */
int bdg_cheb_moments(bdg_t *sys, int kind, int32_t n_cols, const int64_t *probe_rows,
                     uint64_t seed, int64_t col_offset, double scale, int32_t n_moments,
                     int reduce, double *mu, int mu_on_device);
/* Several GPUs, one process (SURVEY 8b / 8e; the reference is single-device, README.md:36-39): sys[g] holds a replica of
 * the SAME Hamiltonian on GPU g (create + scatter it on each; one handle per device).  The n_cols start columns -- probe
 * rows, or Rademacher columns 0 .. n_cols-1 of `seed` -- are split contiguously over the GPUs (the first n_cols %% n_gpu
 * shards take one more), every GPU runs its recursion without communication, and ONE NCCL collective on the handles'
 * streams combines the result: all-reduce of the summed moments (BDG_MU_SUM: mu[n_moments]) or all-gather of the
 * per-column ones (BDG_MU_PER_COLUMN: mu[n_moments][n_cols], columns in their original order).  mu is a host buffer.
 * NCCL is loaded at run time (libnccl.so.2, or $BDG_NCCL_LIB); the communicators of a device list are created on
 * first use and kept (bdg_multi_release destroys them).  n_gpu = 1 is bdg_cheb_moments. */
int bdg_cheb_moments_multi(bdg_t **sys, int n_gpu, int kind, int64_t n_cols, const int64_t *probe_rows,
                           uint64_t seed, double scale, int32_t n_moments, int reduce, double *mu);
int bdg_multi_release(void);
/* Copy the current T_n ([4N, n_cols] row-major complex128) to the host (testing / debugging). */
int bdg_cheb_vectors(bdg_t *sys, int which /*0 = T_n, 1 = T_{n-1}*/, double *out);
/* Algorithmic bytes of one step at the current configuration (SURVEY 8d formula) and the
 * number of blocks after eliminate_zeros. */
int bdg_cheb_info(bdg_t *sys, int64_t *n_blocks, int64_t *bytes_per_step, int32_t *panel_width,
                  int32_t *n_panels, int64_t *launches);
/* What the current recursion actually runs on: *kernel = the BDG_KERNEL_* in use (AUTO resolved),
 * *matrix_bytes_per_step = bytes of matrix data one step reads in that format (blocks or table +
 * codes + indices), *n_distinct_blocks = size of the block dictionary (0 if none was built). */
int bdg_cheb_format(bdg_t *sys, int32_t *kernel, int64_t *matrix_bytes_per_step, int64_t *n_distinct_blocks);
/* Which recursion kernels the current recursion has launched since bdg_cheb_begin (testing): their names as
 * cudaFuncGetName reports them, newline-separated, each once, in the order of their first launch.  *needed = bytes of
 * the NUL-terminated list; names = NULL only sets it, otherwise capacity must be >= *needed.  Host-side bookkeeping. */
int bdg_cheb_launched(bdg_t *sys, char *names, int64_t capacity, int64_t *needed);
int bdg_cheb_end(bdg_t *sys);

/* ---- observables from the moments of the current recursion, evaluated on the device ----------
 *      (consumers: ldos() bodge/hamiltonian.py:349-382, free_energy() bodge/hamiltonian.py:305-319) */
/* g[c * n_z + e] = pref[e] * sum_{n < n_moments} (2 - delta_n0) mu_n[c] w[e]^n   (complex, interleaved).
 * With w = exp(-i arccos z), |w| < 1, and pref = -i / sin(arccos z) this is the resolvent diagonal
 * <x_c| (z - H/scale)^-1 |x_c>: all energies of an LDOS curve for all probe columns in one launch. */
int bdg_kpm_resolvent(bdg_t *sys, int32_t n_moments, int32_t n_z, const double *w, const double *pref,
                      double *g, int g_on_device);
/* out[c] = sum_n coef[n] mu_n[c]  (BDG_MU_PER_COLUMN) or the sum of that over this GPU's columns
 * (BDG_MU_SUM, one double): e.g. coef = Chebyshev coefficients of the free-energy density. */
int bdg_kpm_contract(bdg_t *sys, int32_t n_moments, const double *coef, int reduce, double *out,
                     int out_on_device);
/* Local accumulator: off-diagonal elements of a matrix function, f(H~) ~ sum_n coef[n] T_n(H~), read while the recursion
 * runs.  Register it right after bdg_cheb_begin with the series coef[0 .. n_coef) and a list of reads (column
 * read_col[r] < n_cols of this recursion, row site read_site[r]); it adds the T_0 and T_1 terms at once, and from then on
 * every launch that writes T_n with n < n_coef adds
 *     acc[r][alpha] += coef[n] * T_n[4 * read_site[r] + alpha][read_col[r]],   alpha = 0..3 (complex),
 * one small kernel per launch (4 * n_reads scattered 16-byte loads) next to the unchanged step kernels.  With probe
 * columns x_c = e_q this is acc[r][alpha] = f(H~)[4 site + alpha, q].  There is no moment doubling: the full series needs
 * n_coef - 1 steps (bdg_cheb_steps).  Works with the PAIR and single-step kernels (AUTO, DICT_DIAG, DICT, ELL, DMMA,
 * FMA); the even-vector recursion (T2, also what AUTO_MOMENTS may choose) does not keep the odd vectors and is refused
 * with BDG_E_INVALID.  bdg_cheb_begin discards the accumulator. */
int bdg_cheb_local_begin(bdg_t *sys, int32_t n_coef, const double *coef, int64_t n_reads, const int32_t *read_col,
                         const int32_t *read_site);
/* out[r][alpha] = acc[r][alpha] as complex (interleaved re, im: n_reads * 8 doubles); out_on_device != 0: out is a device
 * pointer on this handle's GPU (e.g. for an NCCL reduce over column shards). */
int bdg_cheb_local_read(bdg_t *sys, double *out, int out_on_device);

#ifdef __cplusplus
}
#endif
#endif /* BDG_H */
