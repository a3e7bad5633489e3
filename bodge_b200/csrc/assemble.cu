// Hamiltonian assembly on the device: BSR skeleton, scatter of the user's 2x2 H/Δ blocks with
// particle-hole + Hermitian fill, Hermiticity check, zero-block compaction, spectral bound.
//
// Replaces bodge/hamiltonian.py:25-170 (reference, pure Python + scipy coo->bsr).  All of it is
// HBM-bound integer / copy work: kernels are one thread per site, per entry element or per
// 16-byte block element with coalesced 128-bit accesses; nothing here is GEMM shaped.
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>

#include "bdg_internal.h"

// ======================================================================================
// errors, memory, handle life cycle
// ======================================================================================
static thread_local char g_error[512] = "";

void bdg_set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof(g_error), fmt, ap);
    va_end(ap);
}

// Device buffers are recycled through a per-device cache: cudaMalloc / cudaFree of the 1.3 GB block array
// cost milliseconds each (page-table work), and the dozen small allocations of a handle another 2-8 ms
// together -- which is what creating or destroying a 10^6-site Hamiltonian spent most of its time on.
// BDG_CACHE_MB bounds the bytes held (0 = off).
namespace {
constexpr int kMaxDevices = 16;
constexpr size_t kCacheMinBytes = 1;  // (small buffers too: a cudaMalloc / cudaFree pair costs more than the few bytes it manages)
std::mutex g_cache_mutex;
std::multimap<size_t, void *> g_cache[kMaxDevices];
size_t g_cache_bytes[kMaxDevices] = {};
std::vector<void *> g_host_pages;  // pinned sizeof(Scalars) pages of destroyed handles

size_t cache_limit() {
    const char *v = getenv("BDG_CACHE_MB");
    return (size_t)(v && *v ? atoll(v) : 8192) << 20;
}

void *cache_take(int device, size_t bytes, size_t *got) {
    if (device < 0 || device >= kMaxDevices || bytes < kCacheMinBytes) return nullptr;
    std::lock_guard<std::mutex> lock(g_cache_mutex);
    auto it = g_cache[device].lower_bound(bytes);
    if (it == g_cache[device].end() || it->first > bytes + bytes / 4) return nullptr;
    void *ptr = it->second;
    *got = it->first;
    g_cache_bytes[device] -= it->first;
    g_cache[device].erase(it);
    return ptr;
}

bool cache_put(int device, void *ptr, size_t bytes) {
    if (device < 0 || device >= kMaxDevices || bytes < kCacheMinBytes) return false;
    std::lock_guard<std::mutex> lock(g_cache_mutex);
    if (g_cache_bytes[device] + bytes > cache_limit()) return false;
    g_cache[device].emplace(bytes, ptr);
    g_cache_bytes[device] += bytes;
    return true;
}

void cache_flush(int device) {
    if (device < 0 || device >= kMaxDevices) return;
    std::lock_guard<std::mutex> lock(g_cache_mutex);
    for (auto &kv : g_cache[device]) cudaFree(kv.second);
    g_cache[device].clear();
    g_cache_bytes[device] = 0;
}
}  // namespace

int dev_alloc(bdg_system *sys, DevBuf &buf, size_t bytes) {
    if (buf.ptr && buf.bytes >= bytes) return BDG_OK;
    dev_free(sys, buf);
    if (bytes == 0) bytes = 16;
    size_t got = bytes;
    void *ptr = cache_take(sys->device, bytes, &got);
    if (!ptr) {
        cudaError_t err = cudaMalloc(&ptr, bytes);
        if (err == cudaErrorMemoryAllocation) {  // give the cached buffers back to the driver and retry
            cudaGetLastError();
            cache_flush(sys->device);
            err = cudaMalloc(&ptr, bytes);
        }
        BDG_CUDA(err);
    }
    buf.ptr = ptr;
    buf.bytes = got;
    sys->dev_bytes += (int64_t)got;
    return BDG_OK;
}

void dev_free(bdg_system *sys, DevBuf &buf) {
    if (buf.ptr) {
        sys->dev_bytes -= (int64_t)buf.bytes;
        bool cached = false;
        if (buf.bytes >= kCacheMinBytes) {
            // cudaFree would wait for the device; a recycled buffer must at least not be in use on this stream
            // (a handle being destroyed has synchronised once already: bdg_destroy)
            if (!sys->quiesced) cudaStreamSynchronize(sys->stream);
            cached = cache_put(sys->device, buf.ptr, buf.bytes);
        }
        if (!cached) cudaFree(buf.ptr);
    }
    buf.ptr = nullptr;
    buf.bytes = 0;
}

extern "C" int bdg_release_cached(int device) {
    BDG_CUDA(cudaSetDevice(device));
    cache_flush(device);
    return BDG_OK;
}

int ensure_scratch(bdg_system *sys, int which, size_t bytes) { return dev_alloc(sys, sys->scratch_i32[which], bytes); }

static void free_bsr(bdg_system *sys, BsrDev &m) {
    dev_free(sys, m.indptr);
    dev_free(sys, m.indices);
    dev_free(sys, m.brow);
    dev_free(sys, m.data);
    m.n_blocks = 0;
}

// Device scalars (mirrored in pinned host memory).
struct Scalars {
    long long first_bad;           // smallest failing entry id (or LLONG_MAX)
    unsigned long long max_bits;   // max of non-negative doubles, compared as integers
    int32_t total;                 // scan totals
    int32_t flag;
};

static int create_common(int device, bdg_system **out) {
    int count = 0;
    cudaError_t err = cudaGetDeviceCount(&count);
    if (err != cudaSuccess || count == 0) {
        bdg_set_error("no CUDA device available (%s)", err == cudaSuccess ? "count = 0" : cudaGetErrorString(err));
        return BDG_E_NO_DEVICE;
    }
    BDG_REQUIRE(device >= 0 && device < count, "device %d out of range (have %d)", device, count);
    BDG_CUDA(cudaSetDevice(device));
    bdg_system *sys = new bdg_system();
    sys->device = device;
    int rc = [&]() -> int {
        BDG_CUDA(cudaDeviceGetAttribute(&sys->sm_count, cudaDevAttrMultiProcessorCount, device));  // (cudaGetDeviceProperties takes milliseconds)
        BDG_CUDA(cudaStreamCreateWithFlags(&sys->own_stream, cudaStreamNonBlocking));
        sys->stream = sys->own_stream;
        BDG_TRY(dev_alloc(sys, sys->scalars, sizeof(Scalars)));
        {   // pinned pages are expensive to create: recycle them like the device buffers
            std::lock_guard<std::mutex> lock(g_cache_mutex);
            if (!g_host_pages.empty()) {
                sys->host_scalars = g_host_pages.back();
                g_host_pages.pop_back();
            }
        }
        if (!sys->host_scalars) BDG_CUDA(cudaMallocHost(&sys->host_scalars, sizeof(Scalars)));
        return BDG_OK;
    }();
    if (rc != BDG_OK) {  // release whatever exists (bdg_destroy copes with a half-built handle)
        bdg_destroy(sys);
        return rc;
    }
    *out = sys;
    return BDG_OK;
}

extern "C" int bdg_abi_version(void) { return BDG_ABI_VERSION; }
extern "C" const char *bdg_last_error(void) { return g_error; }

extern "C" int bdg_device_count(int *count) {
    BDG_REQUIRE(count != nullptr, "null output");
    cudaError_t err = cudaGetDeviceCount(count);
    if (err != cudaSuccess) {
        *count = 0;
        bdg_set_error("cudaGetDeviceCount: %s", cudaGetErrorString(err));
        return BDG_E_NO_DEVICE;
    }
    return BDG_OK;
}

extern "C" int bdg_destroy(bdg_t *sys) {
    if (!sys) return BDG_OK;
    cudaSetDevice(sys->device);
    cudaStreamSynchronize(sys->stream);
    if (sys->own_stream && sys->stream != sys->own_stream) cudaStreamSynchronize(sys->own_stream);
    sys->quiesced = true;  // nothing is enqueued from here on: the buffers go back to the cache without further syncs
    cheb_release(sys);
    free_bsr(sys, sys->skel);
    free_bsr(sys, sys->packed);
    for (auto &b : sys->scratch_i32) dev_free(sys, b);
    for (auto &b : sys->stage) dev_free(sys, b);
    dev_free(sys, sys->pack_flags);
    dev_free(sys, sys->pack_pos);
    dev_free(sys, sys->multi_send);
    dev_free(sys, sys->multi_recv);
    dev_free(sys, sys->scalars);
    if (sys->host_scalars) {
        std::lock_guard<std::mutex> lock(g_cache_mutex);
        g_host_pages.push_back(sys->host_scalars);
    }
    if (sys->own_stream) cudaStreamDestroy(sys->own_stream);
    delete sys;
    return BDG_OK;
}

extern "C" int bdg_set_stream(bdg_t *sys, void *stream) {
    BDG_ENTER(sys);
    BDG_CUDA(cudaStreamSynchronize(sys->stream));
    sys->stream = stream ? static_cast<cudaStream_t>(stream) : sys->own_stream;
    return BDG_OK;
}

extern "C" int bdg_sync(bdg_t *sys) {
    BDG_ENTER(sys);
    BDG_CUDA(cudaStreamSynchronize(sys->stream));
    return BDG_OK;
}

extern "C" int bdg_device_bytes(bdg_t *sys, int64_t *bytes) {
    BDG_REQUIRE(sys && bytes, "null argument");
    *bytes = sys->dev_bytes;
    return BDG_OK;
}

extern "C" int bdg_pinned_alloc(int64_t bytes, void **out) {
    BDG_REQUIRE(out && bytes >= 0, "bad argument");
    BDG_CUDA(cudaMallocHost(out, (size_t)(bytes > 0 ? bytes : 16)));
    return BDG_OK;
}

extern "C" int bdg_pinned_free(void *ptr) {
    if (ptr) BDG_CUDA(cudaFreeHost(ptr));
    return BDG_OK;
}

// ======================================================================================
// small device helpers
// ======================================================================================
namespace {

constexpr int kThreads = 256;

// Position of block column j in block row i, or -1.  Rows are sorted; lattice rows hold <= 7
// entries so a linear scan wins, long rows (generic lattices) fall back to bisection.
__device__ __forceinline__ int find_block(const int32_t *__restrict__ indptr,
                                          const int32_t *__restrict__ indices, int i, int j) {
    int lo = indptr[i], hi = indptr[i + 1];
    if (hi - lo > 16) {
        while (hi - lo > 16) {
            int mid = (lo + hi) >> 1;
            if (indices[mid] <= j) lo = mid; else hi = mid;
        }
    }
    for (int p = lo; p < hi; ++p)
        if (indices[p] == j) return p;
    return -1;
}

__device__ __forceinline__ unsigned long long warp_max_u64(unsigned long long v) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        unsigned long long o = __shfl_xor_sync(0xffffffffu, v, d);
        v = o > v ? o : v;
    }
    return v;
}

// Non-negative doubles (and NaN, which sorts above +inf) order like their bit patterns.
__device__ __forceinline__ void atomic_max_nonneg(unsigned long long *addr, double v) {
    unsigned long long bits = warp_max_u64((unsigned long long)__double_as_longlong(v));
    if ((threadIdx.x & 31) == 0 && bits != 0ull) atomicMax(addr, bits);
}

// ======================================================================================
// cubic skeleton
// ======================================================================================
// Sorted, de-duplicated block columns of `site` on the periodic stencil of an (Lx,Ly,Lz) cubic
// lattice: self plus the +-1 neighbours (with wrap-around) along every axis longer than 1.
// This is the union of lattice.sites(), bonds() and edges() as the reference inserts them
// (hamiltonian.py:47-57): an axis of length 2 gives the same pair as bond and edge, an axis of
// length 1 gives a self pair; both collapse under de-duplication.
__device__ __forceinline__ int cubic_row(int site, int Lx, int Ly, int Lz, int (&cols)[7]) {
    const int z = site % Lz;
    const int y = (site / Lz) % Ly;
    const int x = site / (Lz * Ly);
    int n = 0;
    cols[n++] = site;
    if (Lx > 1) {
        const int s = Ly * Lz;
        cols[n++] = site + (x == 0 ? (Lx - 1) * s : -s);
        cols[n++] = site + (x == Lx - 1 ? -(Lx - 1) * s : s);
    }
    if (Ly > 1) {
        cols[n++] = site + (y == 0 ? (Ly - 1) * Lz : -Lz);
        cols[n++] = site + (y == Ly - 1 ? -(Ly - 1) * Lz : Lz);
    }
    if (Lz > 1) {
        cols[n++] = site + (z == 0 ? (Lz - 1) : -1);
        cols[n++] = site + (z == Lz - 1 ? -(Lz - 1) : 1);
    }
    // insertion sort in registers (n <= 7), then unique
#pragma unroll
    for (int a = 1; a < 7; ++a) {
        if (a < n) {
            int v = cols[a];
            int b = a;
#pragma unroll
            for (int s = 0; s < 6; ++s) {
                if (b > 0 && cols[b - 1] > v) {
                    cols[b] = cols[b - 1];
                    --b;
                }
            }
            cols[b] = v;
        }
    }
    int m = 1;
#pragma unroll
    for (int a = 1; a < 7; ++a) {
        if (a < n && cols[a] != cols[m - 1]) cols[m++] = cols[a];
    }
    return m;
}

__global__ void __launch_bounds__(kThreads) cubic_count(int n_sites, int Lx, int Ly, int Lz,
                                                        int32_t *__restrict__ counts) {
    int site = blockIdx.x * kThreads + threadIdx.x;
    if (site >= n_sites) return;
    int cols[7];
    counts[site] = cubic_row(site, Lx, Ly, Lz, cols);
}

__global__ void __launch_bounds__(kThreads) cubic_fill(int n_sites, int Lx, int Ly, int Lz,
                                                       const int32_t *__restrict__ indptr,
                                                       int32_t *__restrict__ indices,
                                                       int32_t *__restrict__ brow) {
    int site = blockIdx.x * kThreads + threadIdx.x;
    if (site >= n_sites) return;
    int cols[7];
    int m = cubic_row(site, Lx, Ly, Lz, cols);
    int p = indptr[site];
#pragma unroll
    for (int a = 0; a < 7; ++a)
        if (a < m) {
            indices[p + a] = cols[a];
            brow[p + a] = site;
        }
}

// ======================================================================================
// generic skeleton: bucket by row (atomic cursor), per-row sort + unique, scan, compact
// ======================================================================================
__global__ void __launch_bounds__(kThreads) pairs_validate_count(int64_t n_pairs, int n_sites,
                                                                 const int32_t *__restrict__ pi,
                                                                 const int32_t *__restrict__ pj,
                                                                 int32_t *__restrict__ counts,
                                                                 long long *first_bad) {
    int64_t e = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (e >= n_pairs) return;
    int i = pi[e], j = pj[e];
    if (i < 0 || i >= n_sites || j < 0 || j >= n_sites) {
        atomicMin(first_bad, (long long)e);
        return;
    }
    atomicAdd(&counts[i], 1);
    if (i != j) atomicAdd(&counts[j], 1);
}

__global__ void __launch_bounds__(kThreads) pairs_bucket(int64_t n_pairs, const int32_t *__restrict__ pi,
                                                         const int32_t *__restrict__ pj,
                                                         const int32_t *__restrict__ row_start,
                                                         int32_t *__restrict__ cursor,
                                                         int32_t *__restrict__ cols) {
    int64_t e = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (e >= n_pairs) return;
    int i = pi[e], j = pj[e];
    cols[row_start[i] + atomicAdd(&cursor[i], 1)] = j;
    if (i != j) cols[row_start[j] + atomicAdd(&cursor[j], 1)] = i;
}

// One thread per row: in-place insertion sort of the row's bucket, then unique.  Buckets hold the
// row's degree times the lattice's duplication factor (4 for the reference's bonds), i.e. tens.
__global__ void __launch_bounds__(kThreads) rows_sort_unique(int n_sites, const int32_t *__restrict__ row_start,
                                                             int32_t *__restrict__ cols,
                                                             int32_t *__restrict__ uniq_counts) {
    int row = blockIdx.x * kThreads + threadIdx.x;
    if (row >= n_sites) return;
    int lo = row_start[row], hi = row_start[row + 1];
    for (int a = lo + 1; a < hi; ++a) {
        int v = cols[a];
        int b = a;
        while (b > lo && cols[b - 1] > v) {
            cols[b] = cols[b - 1];
            --b;
        }
        cols[b] = v;
    }
    int m = lo;
    for (int a = lo; a < hi; ++a)
        if (a == lo || cols[a] != cols[m - 1]) cols[m++] = cols[a];
    uniq_counts[row] = m - lo;
}

__global__ void __launch_bounds__(kThreads) rows_compact(int n_sites, const int32_t *__restrict__ row_start,
                                                         const int32_t *__restrict__ cols,
                                                         const int32_t *__restrict__ indptr,
                                                         int32_t *__restrict__ indices,
                                                         int32_t *__restrict__ brow) {
    int row = blockIdx.x * kThreads + threadIdx.x;
    if (row >= n_sites) return;
    int src = row_start[row], dst = indptr[row], m = indptr[row + 1] - dst;
    for (int a = 0; a < m; ++a) {
        indices[dst + a] = cols[src + a];
        brow[dst + a] = row;
    }
}

// ======================================================================================
// lookup + scatter + Hermitian check
// ======================================================================================
// kind 0: lookup only (k1).  kind 1: pairing entries need (i,j) and (j,i).
__global__ void __launch_bounds__(kThreads) entries_lookup(int64_t n, int64_t id_base, int n_sites,
                                                           const int32_t *__restrict__ ei,
                                                           const int32_t *__restrict__ ej,
                                                           const int32_t *__restrict__ indptr,
                                                           const int32_t *__restrict__ indices,
                                                           int both, int32_t *__restrict__ k1,
                                                           int32_t *__restrict__ k2, long long *first_bad,
                                                           long long *first_oob) {
    int64_t e = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (e >= n) return;
    int i = ei[e], j = ej[e];
    if (i < 0 || i >= n_sites || j < 0 || j >= n_sites) {
        atomicMin(first_oob, (long long)(id_base + e));
        atomicMin(first_bad, (long long)(id_base + e));
        k1[e] = -1;
        if (both) k2[e] = -1;
        return;
    }
    int a = find_block(indptr, indices, i, j);
    int b = both ? find_block(indptr, indices, j, i) : 0;
    k1[e] = a;
    if (both) k2[e] = b;
    if (a < 0 || b < 0) atomicMin(first_bad, (long long)(id_base + e));
}

// Four threads per entry, one per element of the user's 2x2 matrix (element (r,c) = t>>1, t&1).
//   hopping: blk(i,j)[r][c] = H[r][c];  blk(i,j)[2+r][2+c] = -conj(H[r][c])      (hamiltonian.py:107-108)
//   pairing: blk(i,j)[r][2+c] = D[r][c]; blk(j,i)[2+c][r]  =  conj(D[r][c])      (hamiltonian.py:117-118)
// Negation / conjugation are sign flips, so values (incl. signed zeros) are exactly the
// reference's: -conj(re + i im) = (-re) + i(+im).
__global__ void __launch_bounds__(kThreads) entries_apply(int64_t n, int64_t id_base, int pairing,
                                                          const int32_t *__restrict__ k1,
                                                          const int32_t *__restrict__ k2,
                                                          const double2 *__restrict__ val,
                                                          double2 *__restrict__ data,
                                                          const long long *__restrict__ first_bad) {
    int64_t t = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    int64_t e = t >> 2;
    if (e >= n || id_base + e >= *first_bad) return;
    const int r = (int)(t & 3) >> 1, c = (int)(t & 1);
    const double2 v = val[e * 4 + (t & 3)];
    if (!pairing) {
        double2 *blk = data + (int64_t)k1[e] * 16;
        blk[r * 4 + c] = v;
        blk[(2 + r) * 4 + (2 + c)] = make_double2(-v.x, v.y);
    } else {
        data[(int64_t)k1[e] * 16 + r * 4 + (2 + c)] = v;
        data[(int64_t)k2[e] * 16 + (2 + c) * 4 + r] = make_double2(v.x, -v.y);
    }
}

// max |M - M^H| element-wise (hamiltonian.py:121): 16 threads per block, thread (a,b) compares
// blk(i,j)[a][b] with conj(blk(j,i)[b][a]).
__global__ void __launch_bounds__(kThreads) hermitian_dev(int64_t n_blocks, const int32_t *__restrict__ indptr,
                                                          const int32_t *__restrict__ indices,
                                                          const int32_t *__restrict__ brow,
                                                          const double2 *__restrict__ data,
                                                          unsigned long long *max_bits) {
    int64_t t = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    int64_t k = t >> 4;
    double dev = 0.0;
    if (k < n_blocks) {
        const int el = (int)(t & 15), a = el >> 2, b = el & 3;
        // The 16 threads of one block form a half-warp; shuffle inside that half only -- the other
        // half may belong to a block past the end (odd block counts) and not be here at all.
        const unsigned half_mask = 0xffffu << (threadIdx.x & 16);
        int kt = 0;
        if (el == 0) kt = find_block(indptr, indices, indices[k], brow[k]);
        kt = __shfl_sync(half_mask, kt, (threadIdx.x & 31) & 16);
        const double2 v = data[k * 16 + el];
        if (kt < 0) {
            dev = hypot(v.x, v.y);  // no transposed partner stored: compare with zero
        } else {
            const double2 w = data[(int64_t)kt * 16 + b * 4 + a];
            dev = hypot(v.x - w.x, v.y + w.y);
        }
    }
    atomic_max_nonneg(max_bits, dev);
}

// The same comparison for a LIST of blocks (the ones a scatter wrote; k < 0 = skip): a change of max|M - M^H| can only
// come from a written block or its transposed partner, and the partner's comparison is this one mirrored.
__global__ void __launch_bounds__(kThreads) hermitian_listed(int64_t n, const int32_t *__restrict__ klist,
                                                             const int32_t *__restrict__ indptr,
                                                             const int32_t *__restrict__ indices,
                                                             const int32_t *__restrict__ brow,
                                                             const double2 *__restrict__ data,
                                                             unsigned long long *max_bits) {
    int64_t t = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    int64_t e = t >> 4;
    double dev = 0.0;
    if (e < n) {
        const int k = klist[e];
        const int el = (int)(t & 15), a = el >> 2, b = el & 3;
        const unsigned half_mask = 0xffffu << (threadIdx.x & 16);
        int kt = 0;
        if (el == 0 && k >= 0) kt = find_block(indptr, indices, indices[k], brow[k]);
        kt = __shfl_sync(half_mask, kt, (threadIdx.x & 31) & 16);
        if (k >= 0) {
            const double2 v = data[(int64_t)k * 16 + el];
            if (kt < 0) {
                dev = hypot(v.x, v.y);
            } else {
                const double2 w = data[(int64_t)kt * 16 + b * 4 + a];
                dev = hypot(v.x - w.x, v.y + w.y);
            }
        }
    }
    atomic_max_nonneg(max_bits, dev);
}

// ======================================================================================
// zero-block elimination (scipy bsr eliminate_zeros) and spectral bound
// ======================================================================================
__global__ void __launch_bounds__(kThreads) flag_nonzero(int64_t n_blocks, const double2 *__restrict__ data,
                                                         int32_t *__restrict__ flags) {
    int64_t t = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    int64_t k = t >> 4;
    bool nz = false;
    if (k < n_blocks) {
        const double2 v = data[t];
        nz = (v.x != 0.0) || (v.y != 0.0);  // NaN != 0 is true, -0.0 != 0 is false, like numpy
    }
    unsigned ballot = __ballot_sync(0xffffffffu, nz);
    if (k < n_blocks && (t & 15) == 0) {
        unsigned half = (threadIdx.x & 16) ? (ballot >> 16) : (ballot & 0xffffu);
        flags[k] = half != 0u;
    }
}

__global__ void __launch_bounds__(kThreads) row_kept_counts(int n_sites, const int32_t *__restrict__ indptr,
                                                            const int32_t *__restrict__ flags,
                                                            int32_t *__restrict__ counts, int32_t *max_count) {
    int row = blockIdx.x * kThreads + threadIdx.x;
    int c = 0;
    if (row < n_sites) {
        for (int p = indptr[row]; p < indptr[row + 1]; ++p) c += flags[p];
        counts[row] = c;
    }
    c = __reduce_max_sync(0xffffffffu, c);
    if ((threadIdx.x & 31) == 0 && c > 0) atomicMax(max_count, c);
}

__global__ void __launch_bounds__(kThreads) compact_blocks(int64_t n_blocks, const int32_t *__restrict__ flags,
                                                           const int32_t *__restrict__ pos,
                                                           const int32_t *__restrict__ indices,
                                                           const double2 *__restrict__ data,
                                                           int32_t *__restrict__ out_indices,
                                                           double2 *__restrict__ out_data) {
    int64_t t = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    int64_t k = t >> 4;
    if (k >= n_blocks || !flags[k]) return;
    const int el = (int)(t & 15);
    const int64_t dst = pos[k];
    out_data[dst * 16 + el] = data[t];
    if (el == 0) out_indices[dst] = indices[k];
}

// One thread per scalar row 4*site + a: sum of |entries| over the row's blocks.
__global__ void __launch_bounds__(kThreads) row_abs_sums(int64_t n_rows, const int32_t *__restrict__ indptr,
                                                         const double2 *__restrict__ data,
                                                         unsigned long long *max_bits) {
    int64_t r = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    double sum = 0.0;
    if (r < n_rows) {
        const int site = (int)(r >> 2), a = (int)(r & 3);
        for (int p = indptr[site]; p < indptr[site + 1]; ++p) {
            const double2 *row = data + (int64_t)p * 16 + a * 4;
#pragma unroll
            for (int b = 0; b < 4; ++b) sum += hypot(row[b].x, row[b].y);
        }
    }
    atomic_max_nonneg(max_bits, sum);
}

inline unsigned grid_for(int64_t n) { return (unsigned)ceil_div(n > 0 ? n : 1, kThreads); }

}  // namespace

// ======================================================================================
// host side of the ABI
// ======================================================================================
static int finish_skeleton(bdg_system *sys, int64_t n_sites, int32_t total_blocks) {
    BsrDev &m = sys->skel;
    m.n_sites = n_sites;
    m.n_blocks = total_blocks;
    BDG_TRY(dev_alloc(sys, m.indices, (size_t)total_blocks * sizeof(int32_t)));
    BDG_TRY(dev_alloc(sys, m.brow, (size_t)total_blocks * sizeof(int32_t)));
    BDG_TRY(dev_alloc(sys, m.data, (size_t)total_blocks * 16 * sizeof(double2)));
    BDG_CUDA(cudaMemsetAsync(m.data.ptr, 0, (size_t)total_blocks * 16 * sizeof(double2), sys->stream));
    sys->packed_valid = false;
    return BDG_OK;
}

static int read_total(bdg_system *sys, int32_t *total) {
    Scalars *d = sys->scalars.as<Scalars>();
    Scalars *h = static_cast<Scalars *>(sys->host_scalars);
    BDG_CUDA(cudaMemcpyAsync(&h->total, &d->total, sizeof(int32_t), cudaMemcpyDeviceToHost, sys->stream));
    BDG_CUDA(cudaStreamSynchronize(sys->stream));
    *total = h->total;
    return BDG_OK;
}

extern "C" int bdg_create_cubic(int device, int32_t Lx, int32_t Ly, int32_t Lz, bdg_t **out) {
    BDG_REQUIRE(out != nullptr, "null output");
    BDG_REQUIRE(Lx >= 1 && Ly >= 1 && Lz >= 1, "lattice extents must be >= 1");
    const int64_t n64 = (int64_t)Lx * Ly * Lz;
    BDG_REQUIRE(n64 * 7 < INT32_MAX, "lattice too large for int32 BSR indices");
    bdg_system *sys = nullptr;
    BDG_TRY(create_common(device, &sys));
    sys->cubic[0] = Lx;
    sys->cubic[1] = Ly;
    sys->cubic[2] = Lz;
    const int n = (int)n64;
    int rc = [&]() -> int {
        BDG_TRY(dev_alloc(sys, sys->skel.indptr, (size_t)(n + 1) * sizeof(int32_t)));
        int32_t *indptr = sys->skel.indptr.as<int32_t>();
        Scalars *d = sys->scalars.as<Scalars>();
        cubic_count<<<grid_for(n), kThreads, 0, sys->stream>>>(n, Lx, Ly, Lz, indptr);
        BDG_TRY(exclusive_scan_i32(sys, indptr, indptr, n, &d->total));
        BDG_CUDA(cudaMemcpyAsync(indptr + n, &d->total, sizeof(int32_t), cudaMemcpyDeviceToDevice, sys->stream));
        int32_t total = 0;
        BDG_TRY(read_total(sys, &total));
        BDG_TRY(finish_skeleton(sys, n, total));
        cubic_fill<<<grid_for(n), kThreads, 0, sys->stream>>>(n, Lx, Ly, Lz, indptr, sys->skel.indices.as<int32_t>(),
                                                              sys->skel.brow.as<int32_t>());
        BDG_CUDA(cudaGetLastError());
        BDG_CUDA(cudaStreamSynchronize(sys->stream));
        return BDG_OK;
    }();
    if (rc != BDG_OK) {
        bdg_destroy(sys);
        return rc;
    }
    *out = sys;
    return BDG_OK;
}

extern "C" int bdg_create_generic(int device, int64_t n_sites, int64_t n_pairs, const int32_t *pair_i,
                                  const int32_t *pair_j, bdg_t **out) {
    BDG_REQUIRE(out != nullptr, "null output");
    BDG_REQUIRE(n_sites >= 1 && n_sites < INT32_MAX, "n_sites out of range");
    BDG_REQUIRE(n_pairs >= 0 && 2 * n_pairs < INT32_MAX, "n_pairs out of range");
    BDG_REQUIRE(n_pairs == 0 || (pair_i && pair_j), "null pair arrays");
    bdg_system *sys = nullptr;
    BDG_TRY(create_common(device, &sys));
    const int n = (int)n_sites;
    int rc = [&]() -> int {
        Scalars *d = sys->scalars.as<Scalars>();
        Scalars *h = static_cast<Scalars *>(sys->host_scalars);
        DevBuf d_i, d_j, cols;
        auto cleanup = [&]() {
            dev_free(sys, d_i);
            dev_free(sys, d_j);
            dev_free(sys, cols);
        };
        int inner = [&]() -> int {
            BDG_TRY(dev_alloc(sys, d_i, (size_t)n_pairs * sizeof(int32_t)));
            BDG_TRY(dev_alloc(sys, d_j, (size_t)n_pairs * sizeof(int32_t)));
            BDG_CUDA(cudaMemcpyAsync(d_i.ptr, pair_i, (size_t)n_pairs * sizeof(int32_t), cudaMemcpyHostToDevice, sys->stream));
            BDG_CUDA(cudaMemcpyAsync(d_j.ptr, pair_j, (size_t)n_pairs * sizeof(int32_t), cudaMemcpyHostToDevice, sys->stream));
            // scratch 0: bucket sizes -> bucket starts [n+1]; scratch 1: cursors / unique counts
            BDG_TRY(ensure_scratch(sys, 0, (size_t)(n + 1) * sizeof(int32_t)));
            BDG_TRY(ensure_scratch(sys, 1, (size_t)(n + 1) * sizeof(int32_t)));
            int32_t *row_start = sys->scratch_i32[0].as<int32_t>();
            int32_t *aux = sys->scratch_i32[1].as<int32_t>();
            BDG_CUDA(cudaMemsetAsync(row_start, 0, (size_t)(n + 1) * sizeof(int32_t), sys->stream));
            BDG_CUDA(cudaMemsetAsync(aux, 0, (size_t)(n + 1) * sizeof(int32_t), sys->stream));
            h->first_bad = INT64_MAX;
            BDG_CUDA(cudaMemcpyAsync(&d->first_bad, &h->first_bad, sizeof(long long), cudaMemcpyHostToDevice, sys->stream));
            pairs_validate_count<<<grid_for(n_pairs), kThreads, 0, sys->stream>>>(
                n_pairs, n, d_i.as<int32_t>(), d_j.as<int32_t>(), row_start, &d->first_bad);
            BDG_CUDA(cudaMemcpyAsync(&h->first_bad, &d->first_bad, sizeof(long long), cudaMemcpyDeviceToHost, sys->stream));
            BDG_CUDA(cudaStreamSynchronize(sys->stream));
            if (h->first_bad != INT64_MAX) {
                bdg_set_error("pair %lld has a site index outside [0, %d)", h->first_bad, n);
                return BDG_E_OUT_OF_BOUNDS;
            }
            BDG_TRY(exclusive_scan_i32(sys, row_start, row_start, n, &d->total));
            BDG_CUDA(cudaMemcpyAsync(row_start + n, &d->total, sizeof(int32_t), cudaMemcpyDeviceToDevice, sys->stream));
            int32_t n_entries = 0;
            BDG_TRY(read_total(sys, &n_entries));
            BDG_TRY(dev_alloc(sys, cols, (size_t)n_entries * sizeof(int32_t)));
            pairs_bucket<<<grid_for(n_pairs), kThreads, 0, sys->stream>>>(
                n_pairs, d_i.as<int32_t>(), d_j.as<int32_t>(), row_start, aux, cols.as<int32_t>());
            rows_sort_unique<<<grid_for(n), kThreads, 0, sys->stream>>>(n, row_start, cols.as<int32_t>(), aux);
            BDG_TRY(dev_alloc(sys, sys->skel.indptr, (size_t)(n + 1) * sizeof(int32_t)));
            int32_t *indptr = sys->skel.indptr.as<int32_t>();
            BDG_TRY(exclusive_scan_i32(sys, aux, indptr, n, &d->total));
            BDG_CUDA(cudaMemcpyAsync(indptr + n, &d->total, sizeof(int32_t), cudaMemcpyDeviceToDevice, sys->stream));
            int32_t total = 0;
            BDG_TRY(read_total(sys, &total));
            BDG_TRY(finish_skeleton(sys, n, total));
            rows_compact<<<grid_for(n), kThreads, 0, sys->stream>>>(n, row_start, cols.as<int32_t>(), indptr,
                                                                    sys->skel.indices.as<int32_t>(),
                                                                    sys->skel.brow.as<int32_t>());
            BDG_CUDA(cudaGetLastError());
            BDG_CUDA(cudaStreamSynchronize(sys->stream));
            return BDG_OK;
        }();
        cleanup();
        return inner;
    }();
    if (rc != BDG_OK) {
        bdg_destroy(sys);
        return rc;
    }
    *out = sys;
    return BDG_OK;
}

extern "C" int bdg_skeleton_sizes(bdg_t *sys, int64_t *n_sites, int64_t *n_blocks) {
    BDG_REQUIRE(sys != nullptr, "null handle");
    if (n_sites) *n_sites = sys->skel.n_sites;
    if (n_blocks) *n_blocks = sys->skel.n_blocks;
    return BDG_OK;
}

// Upload entry lists into the handle's staging buffers: stage[0..2] = i, j, values of the list,
// stage[3..4] = k1, k2.
static int stage_entries(bdg_system *sys, int slot, int64_t n, const int32_t *ei, const int32_t *ej,
                         const double *val) {
    DevBuf *st = sys->stage + slot * 5;
    BDG_TRY(dev_alloc(sys, st[0], (size_t)n * sizeof(int32_t)));
    BDG_TRY(dev_alloc(sys, st[1], (size_t)n * sizeof(int32_t)));
    BDG_TRY(dev_alloc(sys, st[3], (size_t)n * sizeof(int32_t)));
    BDG_TRY(dev_alloc(sys, st[4], (size_t)n * sizeof(int32_t)));
    BDG_CUDA(cudaMemcpyAsync(st[0].ptr, ei, (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice, sys->stream));
    BDG_CUDA(cudaMemcpyAsync(st[1].ptr, ej, (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice, sys->stream));
    if (val) {
        BDG_TRY(dev_alloc(sys, st[2], (size_t)n * 4 * sizeof(double2)));
        BDG_CUDA(cudaMemcpyAsync(st[2].ptr, val, (size_t)n * 4 * sizeof(double2), cudaMemcpyHostToDevice, sys->stream));
    }
    return BDG_OK;
}

static int reset_scalars(bdg_system *sys) {
    Scalars *h = static_cast<Scalars *>(sys->host_scalars);
    h->first_bad = INT64_MAX;
    h->max_bits = 0ull;
    h->total = 0;
    h->flag = 0;
    BDG_CUDA(cudaMemcpyAsync(sys->scalars.ptr, h, sizeof(Scalars), cudaMemcpyHostToDevice, sys->stream));
    return BDG_OK;
}

static int fetch_scalars(bdg_system *sys) {
    BDG_CUDA(cudaMemcpyAsync(sys->host_scalars, sys->scalars.ptr, sizeof(Scalars), cudaMemcpyDeviceToHost, sys->stream));
    BDG_CUDA(cudaStreamSynchronize(sys->stream));
    return BDG_OK;
}

extern "C" int bdg_lookup(bdg_t *sys, int64_t n, const int32_t *i, const int32_t *j, int64_t *k,
                          int64_t *bad_entry) {
    BDG_ENTER(sys);
    BDG_REQUIRE(n >= 0 && (n == 0 || (i && j && k)), "bad arguments");
    if (bad_entry) *bad_entry = -1;
    if (n == 0) return BDG_OK;
    Scalars *d = sys->scalars.as<Scalars>();
    Scalars *h = static_cast<Scalars *>(sys->host_scalars);
    BDG_TRY(stage_entries(sys, 0, n, i, j, nullptr));
    BDG_TRY(reset_scalars(sys));
    DevBuf *st = sys->stage;
    // first_oob lives in max_bits' slot for this call (unused otherwise here)
    BDG_CUDA(cudaMemcpyAsync(&d->max_bits, &h->first_bad, sizeof(long long), cudaMemcpyHostToDevice, sys->stream));
    entries_lookup<<<grid_for(n), kThreads, 0, sys->stream>>>(
        n, 0, (int)sys->skel.n_sites, st[0].as<int32_t>(), st[1].as<int32_t>(), sys->skel.indptr.as<int32_t>(),
        sys->skel.indices.as<int32_t>(), 0, st[3].as<int32_t>(), nullptr, &d->first_bad,
        reinterpret_cast<long long *>(&d->max_bits));
    BDG_CUDA(cudaGetLastError());
    std::vector<int32_t> tmp((size_t)n);
    BDG_CUDA(cudaMemcpyAsync(tmp.data(), st[3].ptr, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, sys->stream));
    BDG_TRY(fetch_scalars(sys));
    for (int64_t e = 0; e < n; ++e) k[e] = tmp[(size_t)e];
    if (h->first_bad != INT64_MAX) {
        if (bad_entry) *bad_entry = h->first_bad;
        if ((long long)h->max_bits == h->first_bad) {
            bdg_set_error("entry %lld: site index out of bounds", h->first_bad);
            return BDG_E_OUT_OF_BOUNDS;
        }
        bdg_set_error("entry %lld: block is not part of the lattice skeleton", h->first_bad);
        return BDG_E_NOT_NEIGHBOUR;
    }
    return BDG_OK;
}

static int hermitian_check(bdg_system *sys, double *max_dev) {
    Scalars *d = sys->scalars.as<Scalars>();
    Scalars *h = static_cast<Scalars *>(sys->host_scalars);
    const BsrDev &m = sys->skel;
    h->max_bits = 0ull;
    BDG_CUDA(cudaMemcpyAsync(&d->max_bits, &h->max_bits, sizeof(unsigned long long), cudaMemcpyHostToDevice, sys->stream));
    hermitian_dev<<<grid_for(m.n_blocks * 16), kThreads, 0, sys->stream>>>(
        m.n_blocks, m.indptr.as<int32_t>(), m.indices.as<int32_t>(), m.brow.as<int32_t>(), m.data.as<double2>(),
        &d->max_bits);
    BDG_CUDA(cudaGetLastError());
    BDG_TRY(fetch_scalars(sys));
    double v;
    memcpy(&v, &h->max_bits, sizeof(double));
    *max_dev = v;
    return BDG_OK;
}

extern "C" int bdg_scatter(bdg_t *sys, int64_t n_hop, const int32_t *h_i, const int32_t *h_j, const double *h_val,
                           int64_t n_pair, const int32_t *p_i, const int32_t *p_j, const double *p_val,
                           double herm_tol, double *max_dev, int64_t *bad_entry) {
    BDG_ENTER(sys);
    BDG_REQUIRE(n_hop >= 0 && n_pair >= 0, "negative entry count");
    BDG_REQUIRE(n_hop == 0 || (h_i && h_j && h_val), "null hopping arrays");
    BDG_REQUIRE(n_pair == 0 || (p_i && p_j && p_val), "null pairing arrays");
    BDG_REQUIRE(n_hop < (INT64_C(1) << 40) && n_pair < (INT64_C(1) << 40), "too many entries");
    if (bad_entry) *bad_entry = -1;
    if (max_dev) *max_dev = 0.0;
    Scalars *d = sys->scalars.as<Scalars>();
    Scalars *h = static_cast<Scalars *>(sys->host_scalars);
    const BsrDev &m = sys->skel;
    // The recursion state is stale from here on; whether the compacted matrix and its kernel-native copies are rebuilt
    // or patched in place is decided once the entries are in (below).
    sys->cheb.active = false;
    const bool was_verified = sys->herm_verified;
    sys->herm_verified = false;
    struct Invalidate {  // every early return leaves the copies marked stale
        bdg_system *s;
        bool armed = true;
        ~Invalidate() {
            if (armed) s->packed_valid = false, cheb_deactivate(s);
        }
    } invalidate{sys};

    BDG_TRY(reset_scalars(sys));
    // reuse `total`+`flag` (8 bytes, aligned) as first_oob
    long long *first_oob = reinterpret_cast<long long *>(&d->total);
    BDG_CUDA(cudaMemcpyAsync(first_oob, &h->first_bad, sizeof(long long), cudaMemcpyHostToDevice, sys->stream));
    if (n_hop) BDG_TRY(stage_entries(sys, 0, n_hop, h_i, h_j, h_val));
    if (n_pair) BDG_TRY(stage_entries(sys, 1, n_pair, p_i, p_j, p_val));
    DevBuf *sh = sys->stage, *sp = sys->stage + 5;
    if (n_hop)
        entries_lookup<<<grid_for(n_hop), kThreads, 0, sys->stream>>>(
            n_hop, 0, (int)m.n_sites, sh[0].as<int32_t>(), sh[1].as<int32_t>(), m.indptr.as<int32_t>(),
            m.indices.as<int32_t>(), 0, sh[3].as<int32_t>(), nullptr, &d->first_bad, first_oob);
    if (n_pair)
        entries_lookup<<<grid_for(n_pair), kThreads, 0, sys->stream>>>(
            n_pair, n_hop, (int)m.n_sites, sp[0].as<int32_t>(), sp[1].as<int32_t>(), m.indptr.as<int32_t>(),
            m.indices.as<int32_t>(), 1, sp[3].as<int32_t>(), sp[4].as<int32_t>(), &d->first_bad, first_oob);
    if (n_hop)
        entries_apply<<<grid_for(n_hop * 4), kThreads, 0, sys->stream>>>(
            n_hop, 0, 0, sh[3].as<int32_t>(), nullptr, sh[2].as<double2>(), m.data.as<double2>(), &d->first_bad);
    if (n_pair)
        entries_apply<<<grid_for(n_pair * 4), kThreads, 0, sys->stream>>>(
            n_pair, n_hop, 1, sp[3].as<int32_t>(), sp[4].as<int32_t>(), sp[2].as<double2>(), m.data.as<double2>(),
            &d->first_bad);
    BDG_CUDA(cudaGetLastError());
    BDG_TRY(fetch_scalars(sys));
    if (h->first_bad != INT64_MAX) {
        long long oob;
        memcpy(&oob, &h->total, sizeof(long long));
        if (bad_entry) *bad_entry = h->first_bad;
        const bool pairing = h->first_bad >= n_hop;
        const long long local = pairing ? h->first_bad - n_hop : h->first_bad;
        if (oob == h->first_bad) {
            bdg_set_error("%s entry %lld: site index out of bounds", pairing ? "pairing" : "hopping", local);
            return BDG_E_OUT_OF_BOUNDS;
        }
        bdg_set_error("%s entry %lld: block is not part of the lattice skeleton", pairing ? "pairing" : "hopping", local);
        return BDG_E_NOT_NEIGHBOUR;
    }
    // Kernel-native copies first (the reference leaves the matrix modified when the Hermitian check raises, and so do
    // they): patch the blocks this call wrote, or mark everything stale.
    // (Worth it for a part of the matrix only: one warp per written block costs more than the rebuild's streaming
    // passes once a quarter of all blocks is rewritten.)
    const bool partial = (n_hop + 2 * n_pair) * 4 <= m.n_blocks;
    {
        bool ok = partial && sys->packed_valid && sys->ell.valid;
        if (ok && n_hop) BDG_TRY(ell_patch(sys, n_hop, sh[3].as<int32_t>(), &ok));
        if (ok && n_pair) BDG_TRY(ell_patch(sys, n_pair, sp[3].as<int32_t>(), &ok));
        if (ok && n_pair) BDG_TRY(ell_patch(sys, n_pair, sp[4].as<int32_t>(), &ok));
        invalidate.armed = !ok;
        if (ok) sys->stats[2] += 1, sys->stats[3] += n_hop + 2 * n_pair;
    }
    if (herm_tol >= 0.0) {
        double dev = 0.0;
        if (partial && was_verified && herm_tol >= sys->herm_tol) {
            // everything else passed this tolerance before and has not changed: look at the written blocks only
            h->max_bits = 0ull;
            BDG_CUDA(cudaMemcpyAsync(&d->max_bits, &h->max_bits, sizeof(unsigned long long), cudaMemcpyHostToDevice, sys->stream));
            auto listed = [&](int64_t n, const int32_t *klist) {
                if (n)
                    hermitian_listed<<<grid_for(n * 16), kThreads, 0, sys->stream>>>(
                        n, klist, m.indptr.as<int32_t>(), m.indices.as<int32_t>(), m.brow.as<int32_t>(), m.data.as<double2>(),
                        &d->max_bits);
            };
            listed(n_hop, sh[3].as<int32_t>());
            listed(n_pair, sp[3].as<int32_t>());
            listed(n_pair, sp[4].as<int32_t>());
            BDG_CUDA(cudaGetLastError());
            BDG_TRY(fetch_scalars(sys));
            memcpy(&dev, &h->max_bits, sizeof(double));
            sys->stats[4] += 1;
        } else {
            BDG_TRY(hermitian_check(sys, &dev));
        }
        if (max_dev) *max_dev = dev;
        if (dev > herm_tol) {  // NaN compares false, like np.max(...) > 1e-6 in the reference
            bdg_set_error("The constructed Hamiltonian is not Hermitian! (max deviation %.3e)", dev);
            return BDG_E_NOT_HERMITIAN;
        }
        sys->herm_verified = true;
        sys->herm_tol = herm_tol;
    }
    return BDG_OK;
}

extern "C" int bdg_stats(bdg_t *sys, int64_t out[5]) {
    BDG_REQUIRE(sys && out, "null argument");
    for (int k = 0; k < 5; ++k) out[k] = sys->stats[k];
    return BDG_OK;
}

extern "C" int bdg_clear(bdg_t *sys) {
    BDG_ENTER(sys);
    cheb_deactivate(sys);
    BDG_CUDA(cudaMemsetAsync(sys->skel.data.ptr, 0, (size_t)sys->skel.n_blocks * 16 * sizeof(double2), sys->stream));
    sys->packed_valid = false;
    sys->herm_verified = false;
    return BDG_OK;
}

extern "C" int bdg_import_data(bdg_t *sys, const double *data) {
    BDG_ENTER(sys);
    BDG_REQUIRE(data != nullptr, "null data");
    cheb_deactivate(sys);
    BDG_CUDA(cudaMemcpyAsync(sys->skel.data.ptr, data, (size_t)sys->skel.n_blocks * 16 * sizeof(double2),
                             cudaMemcpyHostToDevice, sys->stream));
    BDG_CUDA(cudaStreamSynchronize(sys->stream));
    sys->packed_valid = false;
    sys->herm_verified = false;
    return BDG_OK;
}

static int fetch_scalars(bdg_system *sys);
// Build sys->packed = skeleton minus all-zero blocks (device resident; also feeds the Chebyshev engine).
int build_packed(bdg_system *sys) {
    if (sys->packed_valid) return BDG_OK;
    const BsrDev &m = sys->skel;
    BsrDev &p = sys->packed;
    Scalars *d = sys->scalars.as<Scalars>();
    const int n = (int)m.n_sites;
    const int64_t nb = m.n_blocks;
    BDG_TRY(dev_alloc(sys, sys->pack_flags, (size_t)(nb + 1) * sizeof(int32_t)));  // kept: a later scatter patches `packed` through them
    BDG_TRY(dev_alloc(sys, sys->pack_pos, (size_t)(nb + 1) * sizeof(int32_t)));
    int32_t *flags = sys->pack_flags.as<int32_t>();
    int32_t *pos = sys->pack_pos.as<int32_t>();
    BDG_TRY(dev_alloc(sys, p.indptr, (size_t)(n + 1) * sizeof(int32_t)));
    int32_t *pptr = p.indptr.as<int32_t>();
    flag_nonzero<<<grid_for(nb * 16), kThreads, 0, sys->stream>>>(nb, m.data.as<double2>(), flags);
    BDG_CUDA(cudaMemsetAsync(&d->flag, 0, sizeof(int32_t), sys->stream));
    row_kept_counts<<<grid_for(n), kThreads, 0, sys->stream>>>(n, m.indptr.as<int32_t>(), flags, pptr, &d->flag);
    BDG_TRY(exclusive_scan_i32(sys, pptr, pptr, n, &d->total));
    BDG_CUDA(cudaMemcpyAsync(pptr + n, &d->total, sizeof(int32_t), cudaMemcpyDeviceToDevice, sys->stream));
    BDG_TRY(exclusive_scan_i32(sys, flags, pos, nb, nullptr));
    int32_t kept = 0;
    BDG_TRY(fetch_scalars(sys));
    kept = static_cast<Scalars *>(sys->host_scalars)->total;
    sys->packed_max_row = static_cast<Scalars *>(sys->host_scalars)->flag;
    p.n_sites = n;
    p.n_blocks = kept;
    BDG_TRY(dev_alloc(sys, p.indices, (size_t)kept * sizeof(int32_t)));
    BDG_TRY(dev_alloc(sys, p.data, (size_t)kept * 16 * sizeof(double2)));
    compact_blocks<<<grid_for(nb * 16), kThreads, 0, sys->stream>>>(nb, flags, pos, m.indices.as<int32_t>(),
                                                                    m.data.as<double2>(), p.indices.as<int32_t>(),
                                                                    p.data.as<double2>());
    BDG_CUDA(cudaGetLastError());
    sys->packed_valid = true;
    sys->stats[0] += 1;
    return BDG_OK;
}

extern "C" int bdg_export_bsr(bdg_t *sys, int eliminate_zeros, int64_t *n_blocks, int32_t *indptr, int32_t *indices,
                              double *data) {
    BDG_ENTER(sys);
    if (eliminate_zeros) BDG_TRY(build_packed(sys));
    const BsrDev &m = eliminate_zeros ? sys->packed : sys->skel;
    if (n_blocks) *n_blocks = m.n_blocks;
    if (indptr)
        BDG_CUDA(cudaMemcpyAsync(indptr, m.indptr.ptr, (size_t)(m.n_sites + 1) * sizeof(int32_t), cudaMemcpyDeviceToHost, sys->stream));
    if (indices && m.n_blocks)
        BDG_CUDA(cudaMemcpyAsync(indices, m.indices.ptr, (size_t)m.n_blocks * sizeof(int32_t), cudaMemcpyDeviceToHost, sys->stream));
    if (data && m.n_blocks)
        BDG_CUDA(cudaMemcpyAsync(data, m.data.ptr, (size_t)m.n_blocks * 16 * sizeof(double2), cudaMemcpyDeviceToHost, sys->stream));
    BDG_CUDA(cudaStreamSynchronize(sys->stream));
    return BDG_OK;
}

// ======================================================================================
// scalar-level exports: matrix("csr") / matrix("csc") / matrix("dense")
// (bodge/hamiltonian.py:144-151: tocsr()/tocsc() + eliminate_zeros(), todense())
// ======================================================================================
// One thread per scalar row (CSR) or scalar column (CSC) of the 4N x 4N matrix.  Entries come
// out in ascending order of the other index, explicit zeros (re == 0 and im == 0; -0.0 is zero,
// NaN is not) are dropped -- what scipy's conversion followed by eliminate_zeros() yields.
// For CSC the blocks of column j are the transposes of the blocks of row j (the skeleton's
// structure is symmetric); their values are fetched from block (i, j).
template <bool FILL>
__global__ void __launch_bounds__(kThreads) scalar_lines(int n_sites, const int32_t *__restrict__ indptr,
                                                         const int32_t *__restrict__ indices,
                                                         const double2 *__restrict__ data, int transpose,
                                                         int32_t *__restrict__ counts,
                                                         const int32_t *__restrict__ offsets,
                                                         int32_t *__restrict__ out_idx, double2 *__restrict__ out_val) {
    const int line = blockIdx.x * kThreads + threadIdx.x;
    if (line >= 4 * n_sites) return;
    const int i = line >> 2, a = line & 3;
    int n = 0;
    int at = FILL ? offsets[line] : 0;
    for (int p = indptr[i]; p < indptr[i + 1]; ++p) {
        const int j = indices[p];
        const int q = transpose ? find_block(indptr, indices, j, i) : p;
        if (q < 0) continue;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const double2 v = data[(size_t)q * 16 + (transpose ? b * 4 + a : a * 4 + b)];
            if (v.x != 0.0 || v.y != 0.0) {
                if (FILL) {
                    out_idx[at] = 4 * j + b;
                    out_val[at] = v;
                    ++at;
                }
                ++n;
            }
        }
    }
    if (!FILL) counts[line] = n;
}

// 16 threads per block: element (a, b) of block (i, j) goes to dense[4i + a][4j + b].
__global__ void __launch_bounds__(kThreads) dense_scatter(int64_t n_blocks, int n_sites,
                                                          const int32_t *__restrict__ brow,
                                                          const int32_t *__restrict__ indices,
                                                          const double2 *__restrict__ data, double2 *__restrict__ out) {
    const int64_t t = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (t >= n_blocks * 16) return;
    const int64_t p = t >> 4;
    const int a = (int)(t >> 2) & 3, b = (int)t & 3;
    // scipy's todense() accumulates into zeros: 0.0 + (-0.0) = +0.0
    const double2 v = data[t];
    out[((size_t)4 * brow[p] + a) * ((size_t)4 * n_sites) + (size_t)4 * indices[p] + b] =
        make_double2(v.x + 0.0, v.y + 0.0);
}

extern "C" int bdg_export_csr(bdg_t *sys, int transpose, int64_t *nnz, int32_t *indptr, int32_t *indices, double *data) {
    BDG_ENTER(sys);
    const BsrDev &m = sys->skel;
    const int n = (int)m.n_sites;
    const int64_t lines = 4 * (int64_t)n;
    Scalars *d = sys->scalars.as<Scalars>();
    BDG_TRY(ensure_scratch(sys, 0, (size_t)(lines + 1) * sizeof(int32_t)));
    int32_t *offsets = sys->scratch_i32[0].as<int32_t>();
    scalar_lines<false><<<grid_for(lines), kThreads, 0, sys->stream>>>(n, m.indptr.as<int32_t>(), m.indices.as<int32_t>(),
                                                                      m.data.as<double2>(), transpose, offsets, nullptr,
                                                                      nullptr, nullptr);
    BDG_CUDA(cudaGetLastError());
    BDG_TRY(exclusive_scan_i32(sys, offsets, offsets, lines, &d->total));
    BDG_CUDA(cudaMemcpyAsync(offsets + lines, &d->total, sizeof(int32_t), cudaMemcpyDeviceToDevice, sys->stream));
    int32_t total = 0;
    BDG_TRY(read_total(sys, &total));
    if (nnz) *nnz = total;
    if (indptr)
        BDG_CUDA(cudaMemcpyAsync(indptr, offsets, (size_t)(lines + 1) * sizeof(int32_t), cudaMemcpyDeviceToHost, sys->stream));
    if (indices && data && total > 0) {
        DevBuf idx, val;
        int rc = dev_alloc(sys, idx, (size_t)total * sizeof(int32_t));
        if (rc == BDG_OK) rc = dev_alloc(sys, val, (size_t)total * sizeof(double2));
        cudaError_t err = cudaSuccess;
        if (rc == BDG_OK) {
            scalar_lines<true><<<grid_for(lines), kThreads, 0, sys->stream>>>(
                n, m.indptr.as<int32_t>(), m.indices.as<int32_t>(), m.data.as<double2>(), transpose, nullptr, offsets,
                idx.as<int32_t>(), val.as<double2>());
            err = cudaGetLastError();
            if (err == cudaSuccess)
                err = cudaMemcpyAsync(indices, idx.ptr, (size_t)total * sizeof(int32_t), cudaMemcpyDeviceToHost, sys->stream);
            if (err == cudaSuccess)
                err = cudaMemcpyAsync(data, val.ptr, (size_t)total * sizeof(double2), cudaMemcpyDeviceToHost, sys->stream);
            if (err == cudaSuccess) err = cudaStreamSynchronize(sys->stream);
        }
        dev_free(sys, idx);
        dev_free(sys, val);
        BDG_TRY(rc);
        BDG_CUDA(err);
    }
    BDG_CUDA(cudaStreamSynchronize(sys->stream));
    return BDG_OK;
}

extern "C" int bdg_export_dense(bdg_t *sys, double *out) {
    BDG_ENTER(sys);
    BDG_REQUIRE(out != nullptr, "null output");
    const BsrDev &m = sys->skel;
    const size_t side = (size_t)4 * m.n_sites;
    const size_t bytes = side * side * sizeof(double2);
    DevBuf dense;
    BDG_TRY(dev_alloc(sys, dense, bytes));
    cudaError_t err = cudaMemsetAsync(dense.ptr, 0, bytes, sys->stream);
    if (err == cudaSuccess && m.n_blocks > 0) {
        dense_scatter<<<grid_for(m.n_blocks * 16), kThreads, 0, sys->stream>>>(
            m.n_blocks, (int)m.n_sites, m.brow.as<int32_t>(), m.indices.as<int32_t>(), m.data.as<double2>(),
            dense.as<double2>());
        err = cudaGetLastError();
    }
    if (err == cudaSuccess) err = cudaMemcpyAsync(out, dense.ptr, bytes, cudaMemcpyDeviceToHost, sys->stream);
    if (err == cudaSuccess) err = cudaStreamSynchronize(sys->stream);
    dev_free(sys, dense);
    BDG_CUDA(err);
    return BDG_OK;
}

extern "C" int bdg_norm_inf(bdg_t *sys, double *norm) {
    BDG_ENTER(sys);
    BDG_REQUIRE(norm != nullptr, "null output");
    Scalars *d = sys->scalars.as<Scalars>();
    Scalars *h = static_cast<Scalars *>(sys->host_scalars);
    const BsrDev &m = sys->skel;
    h->max_bits = 0ull;
    BDG_CUDA(cudaMemcpyAsync(&d->max_bits, &h->max_bits, sizeof(unsigned long long), cudaMemcpyHostToDevice, sys->stream));
    row_abs_sums<<<grid_for(m.n_sites * 4), kThreads, 0, sys->stream>>>(m.n_sites * 4, m.indptr.as<int32_t>(),
                                                                        m.data.as<double2>(), &d->max_bits);
    BDG_CUDA(cudaGetLastError());
    BDG_TRY(fetch_scalars(sys));
    memcpy(norm, &h->max_bits, sizeof(double));
    return BDG_OK;
}
