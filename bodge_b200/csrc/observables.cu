// Observables from the Chebyshev moments, evaluated on the device where the moments already
// live (SURVEY 8f-1): the resolvent diagonal behind ldos() (reference bodge/hamiltonian.py:349-382
// solves (eps + i Gamma - H) X = B with SuperLU per energy) and series contractions
// sum_n c_n mu_n behind free_energy() (reference bodge/hamiltonian.py:305-319).
//
// Moments are never materialised: mu_n[c] is read straight from the per-step dot products
// (moment doubling: mu_n = 2 dots[n] - mu_{n mod 2} for n >= 2).
#include "bdg_internal.h"

namespace {

constexpr int kObsThreads = 128;

__device__ __forceinline__ double moment(const double *__restrict__ dots, int n, int stride, int c, double mu0, double mu1) {
    if (n == 0) return mu0;
    if (n == 1) return mu1;
    return 2.0 * dots[(size_t)n * stride + c] - ((n & 1) ? mu1 : mu0);
}

// g[c][e] = pref[e] * sum_n (2 - delta_n0) mu_n[c] w[e]^n   (Horner from the top; |w| < 1)
// With w = exp(-i arccos z) on the decaying branch and pref = -i / sin(arccos z) this is
// <x_c| (z - H~)^-1 |x_c>  (kpm.resolvent_diagonal).  Threads: column fastest (coalesced dots).
__global__ void __launch_bounds__(kObsThreads)
kpm_resolvent(const double *__restrict__ dots, int n_moments, int n_cols, int stride, int n_z,
              const double2 *__restrict__ w, const double2 *__restrict__ pref, double2 *__restrict__ g) {
    const int64_t t = (int64_t)blockIdx.x * kObsThreads + threadIdx.x;
    if (t >= (int64_t)n_cols * n_z) return;
    const int c = (int)(t % n_cols), e = (int)(t / n_cols);
    const double mu0 = dots[c], mu1 = dots[stride + c];
    const double2 ww = w[e];
    double ar = 0.0, ai = 0.0;
    for (int n = n_moments - 1; n >= 0; --n) {
        const double m = (n == 0 ? 1.0 : 2.0) * moment(dots, n, stride, c, mu0, mu1);
        const double nr = ar * ww.x - ai * ww.y + m;
        ai = ar * ww.y + ai * ww.x;
        ar = nr;
    }
    const double2 p = pref[e];
    g[(size_t)c * n_z + e] = make_double2(p.x * ar - p.y * ai, p.x * ai + p.y * ar);
}

// out[c] = sum_n coef[n] mu_n[c]; one warp per column, lanes stride over n, fixed-order shuffle
// reduction (deterministic).
__global__ void __launch_bounds__(kObsThreads)
kpm_contract(const double *__restrict__ dots, int n_moments, int n_cols, int stride, const double *__restrict__ coef,
             double *__restrict__ out) {
    const int c = (blockIdx.x * kObsThreads + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (c >= n_cols) return;
    const double mu0 = dots[c], mu1 = dots[stride + c];
    double s = 0.0;
    for (int n = lane; n < n_moments; n += 32) s += coef[n] * moment(dots, n, stride, c, mu0, mu1);
#pragma unroll
    for (int d = 16; d; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
    if (lane == 0) out[c] = s;
}

// acc[r][alpha] += ca * x_a[off[r] + alpha] (+ cb * x_b[...]): one thread per (read, alpha), each owning its
// accumulator element, so the sum runs in the order of n on every configuration.  Off-diagonal elements
// <e_row| T_n |x_c> have no moment doubling: every term is read from its own vector.
__global__ void __launch_bounds__(kObsThreads)
local_accumulate_kernel(const double2 *__restrict__ x_a, const double2 *__restrict__ x_b, double ca, double cb,
                        const int64_t *__restrict__ off, int64_t n_reads, double2 *__restrict__ acc) {
    const int64_t t = (int64_t)blockIdx.x * kObsThreads + threadIdx.x;
    if (t >= 4 * n_reads) return;
    const int64_t o = off[t >> 2] + (t & 3);
    double2 s = acc[t];
    const double2 a = x_a[o];
    s.x += ca * a.x;
    s.y += ca * a.y;
    if (x_b) {
        const double2 b = x_b[o];
        s.x += cb * b.x;
        s.y += cb * b.y;
    }
    acc[t] = s;
}

__global__ void sum_columns(const double *__restrict__ in, int n, double *__restrict__ out) {
    // single warp, fixed order
    double s = 0.0;
    for (int i = threadIdx.x; i < n; i += 32) s += in[i];
#pragma unroll
    for (int d = 16; d; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
    if (threadIdx.x == 0) out[0] = s;
}

}  // namespace

static int check_active(bdg_system *sys, int32_t n_moments) {
    const ChebState &st = sys->cheb;
    BDG_REQUIRE(st.active, "bdg_cheb_begin has not been called");
    BDG_REQUIRE(n_moments >= 1 && n_moments <= 2 * (st.steps_done + 1), "only %d moments available, %d requested",
                2 * (st.steps_done + 1), n_moments);
    return t2_finish_dots(sys);  // (the even-vector recursion leaves its dot rows in another form)
}

extern "C" int bdg_kpm_resolvent(bdg_t *sys, int32_t n_moments, int32_t n_z, const double *w, const double *pref,
                                 double *g, int g_on_device) {
    BDG_ENTER(sys);
    BDG_TRY(check_active(sys, n_moments));
    BDG_REQUIRE(n_z >= 1 && w && pref && g, "null or empty argument");
    ChebState &st = sys->cheb;
    const size_t zbytes = (size_t)n_z * sizeof(double2);
    const size_t count = (size_t)st.n_cols * n_z;
    // obs_tmp = [w | pref | g]
    BDG_TRY(dev_alloc(sys, st.obs_tmp, 2 * zbytes + (g_on_device ? 0 : count * sizeof(double2))));
    double2 *dw = st.obs_tmp.as<double2>(), *dp = dw + n_z;
    double2 *dg = g_on_device ? reinterpret_cast<double2 *>(g) : dp + n_z;
    BDG_CUDA(cudaMemcpyAsync(dw, w, zbytes, cudaMemcpyHostToDevice, sys->stream));
    BDG_CUDA(cudaMemcpyAsync(dp, pref, zbytes, cudaMemcpyHostToDevice, sys->stream));
    kpm_resolvent<<<(unsigned)ceil_div((int64_t)count, kObsThreads), kObsThreads, 0, sys->stream>>>(
        st.dots.as<double>(), n_moments, st.n_cols, st.n_panels * st.panel_width, n_z, dw, dp, dg);
    BDG_CUDA(cudaGetLastError());
    st.launches += 1;
    if (!g_on_device)
        BDG_CUDA(cudaMemcpyAsync(g, dg, count * sizeof(double2), cudaMemcpyDeviceToHost, sys->stream));
    BDG_CUDA(cudaStreamSynchronize(sys->stream));  // w / pref are borrowed only for this call
    return BDG_OK;
}

extern "C" int bdg_kpm_contract(bdg_t *sys, int32_t n_moments, const double *coef, int reduce, double *out,
                                int out_on_device) {
    BDG_ENTER(sys);
    BDG_TRY(check_active(sys, n_moments));
    BDG_REQUIRE(coef && out, "null argument");
    BDG_REQUIRE(reduce == BDG_MU_PER_COLUMN || reduce == BDG_MU_SUM, "unknown reduce mode");
    ChebState &st = sys->cheb;
    const int k = st.n_cols;
    // obs_tmp = [coef | per-column | total]
    BDG_TRY(dev_alloc(sys, st.obs_tmp, ((size_t)n_moments + k + 1) * sizeof(double)));
    double *dc = st.obs_tmp.as<double>(), *dcol = dc + n_moments, *dtot = dcol + k;
    BDG_CUDA(cudaMemcpyAsync(dc, coef, (size_t)n_moments * sizeof(double), cudaMemcpyHostToDevice, sys->stream));
    double *col_dst = (!reduce && out_on_device) ? out : dcol;
    kpm_contract<<<(unsigned)ceil_div((int64_t)k * 32, kObsThreads), kObsThreads, 0, sys->stream>>>(
        st.dots.as<double>(), n_moments, k, st.n_panels * st.panel_width, dc, col_dst);
    BDG_CUDA(cudaGetLastError());
    st.launches += 1;
    const double *src = col_dst;
    size_t n_out = (size_t)k;
    if (reduce) {
        double *tot_dst = out_on_device ? out : dtot;
        sum_columns<<<1, 32, 0, sys->stream>>>(dcol, k, tot_dst);
        BDG_CUDA(cudaGetLastError());
        st.launches += 1;
        src = tot_dst;
        n_out = 1;
    }
    if (!out_on_device)
        BDG_CUDA(cudaMemcpyAsync(out, src, n_out * sizeof(double), cudaMemcpyDeviceToHost, sys->stream));
    BDG_CUDA(cudaStreamSynchronize(sys->stream));
    return BDG_OK;
}

int local_accumulate(bdg_system *sys, int n, const void *x_a, const void *x_b) {
    ChebState &st = sys->cheb;
    const int n_coef = (int)st.local_coef.size();
    if (!st.local || n >= n_coef) return BDG_OK;
    const bool second = x_b && n + 1 < n_coef;
    local_accumulate_kernel<<<(unsigned)ceil_div(4 * st.local_reads, kObsThreads), kObsThreads, 0, sys->stream>>>(
        static_cast<const double2 *>(x_a), second ? static_cast<const double2 *>(x_b) : nullptr, st.local_coef[n],
        second ? st.local_coef[n + 1] : 0.0, st.local_off.as<int64_t>(), st.local_reads, st.local_acc.as<double2>());
    BDG_CUDA(cudaGetLastError());
    st.launches += 1;
    return BDG_OK;
}

extern "C" int bdg_cheb_local_begin(bdg_t *sys, int32_t n_coef, const double *coef, int64_t n_reads, const int32_t *read_col,
                                    const int32_t *read_site) {
    BDG_ENTER(sys);
    ChebState &st = sys->cheb;
    BDG_REQUIRE(st.active, "bdg_cheb_begin has not been called");
    BDG_REQUIRE(!st.even(),
                "the even-vector recursion (kernel T2) keeps only every second Chebyshev vector, so it cannot accumulate "
                "local matrix elements of a series: begin the recursion with the pair or a single-step kernel");
    BDG_REQUIRE(st.steps_done == 0, "register the local accumulator right after bdg_cheb_begin (%d steps already taken)",
                st.steps_done);
    BDG_REQUIRE(n_coef >= 1 && coef, "need at least one coefficient");
    BDG_REQUIRE(n_reads >= 1 && read_col && read_site, "need at least one read");
    const int64_t n_sites = sys->packed.n_sites;
    const int pw = st.panel_width;
    std::vector<int64_t> off((size_t)n_reads);
    for (int64_t r = 0; r < n_reads; ++r) {
        const int32_t c = read_col[r], s = read_site[r];
        BDG_REQUIRE(c >= 0 && c < st.n_cols, "read %lld: column %d outside [0, %d)", (long long)r, c, st.n_cols);
        BDG_REQUIRE(s >= 0 && s < n_sites, "read %lld: site %d outside [0, %lld)", (long long)r, s, (long long)n_sites);
        off[(size_t)r] = (((int64_t)(c / pw) * n_sites + s) * pw + c % pw) * 4;
    }
    BDG_TRY(dev_alloc(sys, st.local_off, (size_t)n_reads * sizeof(int64_t)));
    BDG_TRY(dev_alloc(sys, st.local_acc, (size_t)n_reads * 4 * sizeof(double2)));
    BDG_CUDA(cudaMemcpyAsync(st.local_off.ptr, off.data(), (size_t)n_reads * sizeof(int64_t), cudaMemcpyHostToDevice,
                             sys->stream));
    BDG_CUDA(cudaMemsetAsync(st.local_acc.ptr, 0, (size_t)n_reads * 4 * sizeof(double2), sys->stream));
    st.local_coef.assign(coef, coef + n_coef);
    st.local_reads = n_reads;
    st.local = true;
    // T_0 is still in vec[prev], T_1 in vec[cur] (bdg_cheb_begin took the first step)
    BDG_TRY(local_accumulate(sys, 0, st.vec[st.prev].ptr, st.vec[st.cur].ptr));
    BDG_CUDA(cudaStreamSynchronize(sys->stream));  // `off` is a local of this call
    return BDG_OK;
}

extern "C" int bdg_cheb_local_read(bdg_t *sys, double *out, int out_on_device) {
    BDG_ENTER(sys);
    ChebState &st = sys->cheb;
    BDG_REQUIRE(st.active && st.local, "no local accumulator on an active recursion (bdg_cheb_local_begin)");
    BDG_REQUIRE(out, "null output");
    BDG_CUDA(cudaMemcpyAsync(out, st.local_acc.ptr, (size_t)st.local_reads * 4 * sizeof(double2),
                             out_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, sys->stream));
    BDG_CUDA(cudaStreamSynchronize(sys->stream));
    return BDG_OK;
}
