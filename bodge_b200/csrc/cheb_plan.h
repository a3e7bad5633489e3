// Stepping planner of the Chebyshev recursion (bdg_cheb_begin, cheb.cu): from what the kernels' copies of the matrix allow,
// which stepping, matrix format and panel width a request runs on, or why it is refused; and the plan switches every planner
// reads.  Host code, internal: tests/cpp/plan_check.cpp checks plan_stepping on the CPU.
#pragma once

#include <algorithm>
#include <cstdlib>

#include "bdg_internal.h"

// Plan switches (INTEGRATION.md): member x_y holds BDG_X_Y.  bdg_cheb_begin reads them once (read_plan_switches, which
// holds the defaults) and plan_stepping and the configure functions plan from this copy, so they hold for the whole
// recursion.  Extents and segment lengths: <= 0 = the planner's; pair_self, cube_shape and the balances: < 0 = the planner's.
struct PlanSwitches {
    bool auto_pair, auto_cube;
    bool ell_sd, ell_walk;
    int ell_pz, ell_seg, ell_prefetch;
    int pair_self, pair_p, pair_seg, pair_balance;
    bool pair_open;
    int cube_shape, cube_seg, cube_balance;
};

// What the matrix copies allow (EllDev, formats.cu) and the lattice the plan runs on.  All false / zero when the request
// needs no copies (DMMA, FMA).
struct PlanFacts {
    bool ell_usable, dict_usable, diag_usable, pair_usable, cube_usable;
    int64_t n_sites;
    int Ly, Lz;  // bdg_system::cubic[1], [2]
    int sm_count;
};

struct SteppingPlan {
    const char *refusal;  // nullptr: accepted; else why the matrix cannot run the requested kernel
    Stepping stepping;
    int format;           // BDG_KERNEL_* of the single-step kernel and of the matrix copies the plan reads (ChebState::kernel)
    int panel_width, n_panels;
};

namespace {

// AUTO runs two steps per pass wherever the DFMA variant of the pair kernel applies: 1.33x the single-step
// dictionary kernel at C5 (profiles/r01/s4_pair_v2.log).  The DMMA variant (complex hopping / pairing on the
// bonds, C3) is FP64-pipe-bound and slower than its single-step kernel, so it stays opt-in.
constexpr bool kAutoPairDefault = true;

// Every plan switch (PlanSwitches), read once per recursion.
inline PlanSwitches read_plan_switches() {
    // BDG_ELL_PZ, BDG_PAIR_P: a set value counts as at least 1; unset or empty: 0
    const auto extent = [](const char *name) {
        const char *v = getenv(name);
        return v && *v ? std::max(1, atoi(v)) : 0;
    };
    PlanSwitches s;
    s.auto_pair = env_int("BDG_AUTO_PAIR", kAutoPairDefault) != 0;
    s.auto_cube = env_int("BDG_AUTO_CUBE", 1) != 0;
    s.ell_sd = env_int("BDG_ELL_SD", 1) != 0;
    s.ell_walk = env_int("BDG_ELL_WALK", 1) != 0;
    s.ell_pz = extent("BDG_ELL_PZ");
    s.ell_seg = env_int("BDG_ELL_SEG", 0);
    s.ell_prefetch = env_int("BDG_ELL_PREFETCH", 1);
    s.pair_self = env_int("BDG_PAIR_SELF", -1);
    s.pair_open = env_int("BDG_PAIR_OPEN", 1) != 0;
    s.pair_p = extent("BDG_PAIR_P");
    s.pair_seg = env_int("BDG_PAIR_SEG", 0);
    s.pair_balance = env_int("BDG_PAIR_BALANCE", -1);
    s.cube_shape = env_int("BDG_CUBE_SHAPE", -1);
    s.cube_seg = env_int("BDG_CUBE_SEG", 0);
    s.cube_balance = env_int("BDG_CUBE_BALANCE", -1);
    return s;
}

// The plan of a recursion of `n_cols` columns asked for with `kernel` (an assigned BDG_KERNEL_*; bdg_cheb_begin refuses the
// others).  AUTO and AUTO_MOMENTS always get a plan; a kernel asked for by name is refused when the matrix cannot run it.
inline SteppingPlan plan_stepping(int kernel, int n_cols, const PlanFacts &f, const PlanSwitches &sw) {
    SteppingPlan plan{nullptr, Stepping::Single, kernel, 0, 0};
    // The pair kernel works on 8-column panels of the dictionary format; single leftover steps
    // (and T_1) run on the single-step dictionary kernel of the same format.
    // The two-step kernels work on 8-column panels.  Fewer than 5 columns (ldos() of one site = 4) are padded to
    // a panel when the vectors are small enough to live in L2 (<= 64 Ki sites: 32 MB per vector): such runs are
    // launch-latency-bound, and two steps per launch halve the launches; at HBM-bound sizes the padding would
    // cost more bytes than the fusion saves, so narrow panels stay on the single-step kernels there.
    const bool small = f.n_sites <= (1 << 16);
    const bool pair_ok = f.pair_usable && (n_cols >= 5 || small);
    // Three-dimensional lattices: the even-vector recursion on 4-column panels (cheb_cube.cu): open stencil,
    // real-diagonal hopping blocks, few distinct blocks (its fragments are held in registers): EllDev::cube_usable.
    const bool cube_ok = f.cube_usable && (n_cols >= 3 || small);
    if (kernel == BDG_KERNEL_PAIR && !pair_ok) {
        plan.refusal = "the two-steps-per-pass kernel needs >= 5 columns (any number on lattices of <= 65536 sites) and a block "
                       "dictionary on a lattice with one-dimensional x-planes and a nearest-neighbour stencil";
        return plan;
    }
    if (kernel == BDG_KERNEL_T2 && !pair_ok && !cube_ok) {
        plan.refusal = "the even-vector recursion needs a block dictionary on a lattice with a nearest-neighbour stencil: one-dimensional "
                       "x-planes and >= 5 columns, or a three-dimensional open lattice with real-diagonal hopping blocks, <= 64 "
                       "distinct blocks and >= 3 columns (any number of columns on lattices of <= 65536 sites)";
        return plan;
    }
    // The two-step kernels pay on every dictionary matrix they take (round 2, profiles/r02/41_* .. 43_*): rows of real-
    // diagonal hopping blocks (DFMA), general hopping blocks next to real-diagonal on-site blocks (SD: d-wave / Rashba
    // models, +12..44 % over the single-step kernel) and rows of ten MMAs (+22..42 % at 8 columns, +24..32 % at >= 64
    // columns on 10^6 sites, level at C3 with 64..512 columns).
    const bool prefer = pair_ok && sw.auto_pair;
    // Callers that only read moments / observables get the even-vector recursion (three vector passes per
    // two steps); callers that step and look at T_n, T_{n-1} the pair kernel (four).
    // ... preferred where its items fill the machine without cutting x into segments (one CTA per SM marches an 8 x 8 patch:
    // C4 = 64 patches x 2 panels); on smaller lattices the single-step kernel's finer grid wins.
    const int64_t cube_items = ceil_div(f.Ly, 8) * ceil_div(f.Lz, 8) * ceil_div(n_cols, 4);
    const bool prefer_cube = cube_ok && sw.auto_cube && 4 * cube_items >= 3 * (int64_t)f.sm_count;
    // (the even-vector recursion without pair_ok has cube_ok: the refusal above, or prefer_cube)
    if (kernel == BDG_KERNEL_T2 || (kernel == BDG_KERNEL_AUTO_MOMENTS && (prefer || prefer_cube)))
        plan.stepping = pair_ok ? Stepping::EvenPlane : Stepping::EvenCube;
    else if (kernel == BDG_KERNEL_PAIR || (kernel == BDG_KERNEL_AUTO && prefer))
        plan.stepping = Stepping::Pair;
    if (kernel == BDG_KERNEL_PAIR || kernel == BDG_KERNEL_T2 || kernel == BDG_KERNEL_AUTO_MOMENTS) kernel = BDG_KERNEL_AUTO;
    if (kernel == BDG_KERNEL_ELL && !f.ell_usable)
        plan.refusal = "the fixed-width (ELL) kernel needs block rows of <= 8 blocks with little padding";
    else if (kernel == BDG_KERNEL_DICT && !f.dict_usable)
        plan.refusal = "the block-dictionary kernel needs a fixed-width matrix whose distinct blocks are few";
    else if (kernel == BDG_KERNEL_DICT_DIAG && !f.diag_usable)
        plan.refusal = "the diagonal-hopping kernel needs a block dictionary whose off-site blocks are real and diagonal";
    if (plan.refusal) return plan;
    if (kernel == BDG_KERNEL_AUTO)
        kernel = f.diag_usable   ? BDG_KERNEL_DICT_DIAG
                 : f.dict_usable ? BDG_KERNEL_DICT
                 : f.ell_usable  ? BDG_KERNEL_ELL
                                 : BDG_KERNEL_DMMA;
    plan.format = kernel;
    plan.panel_width = plan.stepping == Stepping::EvenCube ? 4
                       : (n_cols >= 5 || plan.stepping != Stepping::Single) ? 8
                                                                           : (n_cols >= 3 ? 4 : n_cols);
    plan.n_panels = (int)ceil_div(n_cols, plan.panel_width);
    return plan;
}

}  // namespace
