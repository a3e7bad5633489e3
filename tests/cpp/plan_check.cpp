// Host-side check of the stepping planner (bodge_b200/csrc/cheb_plan.h), built and run by tests/test_plan.py.  Over every
// consistent set of matrix facts, every assigned kernel number, column counts, lattice sizes on both sides of the 64 Ki-site
// rule and lattice cross-sections on both sides of the rule that prefers the three-dimensional kernel, and both auto
// switches, plan_stepping must:
//   - refuse exactly when the documented condition fails, with the message bdg_cheb_begin reports, word for word;
//   - never refuse AUTO or AUTO_MOMENTS;
//   - pick the stepping and the format the rules give, and never one whose flag is false;
//   - cut the columns into panels of 4 (EvenCube), 8 (Pair, EvenPlane) or the single-step width.
// Then the plans of the bench systems under the default switches.  No device code runs.
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "cheb_plan.h"

static const char *const kPairRefusal =
    "the two-steps-per-pass kernel needs >= 5 columns (any number on lattices of <= 65536 sites) and a block dictionary on a "
    "lattice with one-dimensional x-planes and a nearest-neighbour stencil";
static const char *const kT2Refusal =
    "the even-vector recursion needs a block dictionary on a lattice with a nearest-neighbour stencil: one-dimensional x-planes "
    "and >= 5 columns, or a three-dimensional open lattice with real-diagonal hopping blocks, <= 64 distinct blocks and >= 3 "
    "columns (any number of columns on lattices of <= 65536 sites)";
static const char *const kEllRefusal = "the fixed-width (ELL) kernel needs block rows of <= 8 blocks with little padding";
static const char *const kDictRefusal = "the block-dictionary kernel needs a fixed-width matrix whose distinct blocks are few";
static const char *const kDiagRefusal =
    "the diagonal-hopping kernel needs a block dictionary whose off-site blocks are real and diagonal";

static const char *name(Stepping s) {
    switch (s) {
        case Stepping::Single: return "Single";
        case Stepping::Pair: return "Pair";
        case Stepping::EvenPlane: return "EvenPlane";
        case Stepping::EvenCube: return "EvenCube";
    }
    return "?";
}

static void fail(const char *what, int kernel, int n_cols, const PlanFacts &f, const PlanSwitches &sw, const SteppingPlan &p) {
    std::printf("FAIL %s: kernel=%d n_cols=%d ell=%d dict=%d diag=%d pair=%d cube=%d n_sites=%lld Ly=%d Lz=%d sm=%d auto_pair=%d "
                "auto_cube=%d -> refusal=%s stepping=%s format=%d panel_width=%d n_panels=%d\n",
                what, kernel, n_cols, f.ell_usable, f.dict_usable, f.diag_usable, f.pair_usable, f.cube_usable, (long long)f.n_sites,
                f.Ly, f.Lz, f.sm_count, sw.auto_pair, sw.auto_cube, p.refusal ? p.refusal : "none", name(p.stepping), p.format,
                p.panel_width, p.n_panels);
    std::exit(1);
}

// The documented rules, restated.
static const char *expected_refusal(int kernel, bool pair_ok, bool cube_ok, const PlanFacts &f) {
    if (kernel == BDG_KERNEL_PAIR && !pair_ok) return kPairRefusal;
    if (kernel == BDG_KERNEL_T2 && !pair_ok && !cube_ok) return kT2Refusal;
    if (kernel == BDG_KERNEL_ELL && !f.ell_usable) return kEllRefusal;
    if (kernel == BDG_KERNEL_DICT && !f.dict_usable) return kDictRefusal;
    if (kernel == BDG_KERNEL_DICT_DIAG && !f.diag_usable) return kDiagRefusal;
    return nullptr;
}

// How often each side of each rule was reached (every count must end up non-zero)
static struct {
    long refused, named;                  // a kernel asked for by name: refused, accepted
    long even_plane, even_cube, declined; // AUTO_MOMENTS: plane, cube, cube_ok but below the cube threshold
    long narrow_pair, narrow_single;      // < 5 columns on a pair-usable lattice: <= 64 Ki sites (pair), more (single step)
} reached;

static void check(int kernel, int n_cols, const PlanFacts &f, const PlanSwitches &sw) {
    const SteppingPlan p = plan_stepping(kernel, n_cols, f, sw);
    const bool small = f.n_sites <= 65536;
    const bool pair_ok = f.pair_usable && (n_cols >= 5 || small);
    const bool cube_ok = f.cube_usable && (n_cols >= 3 || small);
    const bool auto_kernel = kernel == BDG_KERNEL_AUTO || kernel == BDG_KERNEL_AUTO_MOMENTS;

    const char *refusal = expected_refusal(kernel, pair_ok, cube_ok, f);
    if (!refusal != !p.refusal) fail(refusal ? "not refused" : "refused", kernel, n_cols, f, sw, p);
    if (refusal && std::strcmp(refusal, p.refusal) != 0) fail("refusal text", kernel, n_cols, f, sw, p);
    if (auto_kernel && p.refusal) fail("AUTO refused", kernel, n_cols, f, sw, p);
    if (refusal) {
        reached.refused += 1;
        return;
    }
    if (!auto_kernel) reached.named += 1;

    // stepping
    const bool prefer = pair_ok && sw.auto_pair;
    const long cube_items = ((f.Ly + 7) / 8) * (long)((f.Lz + 7) / 8) * ((n_cols + 3) / 4);
    const bool prefer_cube = cube_ok && sw.auto_cube && 4 * cube_items >= 3L * f.sm_count;
    Stepping want = Stepping::Single;
    if (kernel == BDG_KERNEL_T2 || (kernel == BDG_KERNEL_AUTO_MOMENTS && (prefer || prefer_cube)))
        want = pair_ok ? Stepping::EvenPlane : Stepping::EvenCube;
    else if (kernel == BDG_KERNEL_PAIR || (kernel == BDG_KERNEL_AUTO && prefer))
        want = Stepping::Pair;
    if (p.stepping != want) fail("stepping", kernel, n_cols, f, sw, p);
    if ((p.stepping == Stepping::Pair || p.stepping == Stepping::EvenPlane) && !pair_ok) fail("two-step plan without pair_ok", kernel, n_cols, f, sw, p);
    if (p.stepping == Stepping::EvenCube && !cube_ok) fail("cube plan without cube_ok", kernel, n_cols, f, sw, p);
    if (kernel == BDG_KERNEL_AUTO_MOMENTS) {
        reached.even_plane += p.stepping == Stepping::EvenPlane;
        reached.even_cube += p.stepping == Stepping::EvenCube;
        reached.declined += cube_ok && sw.auto_cube && !pair_ok && p.stepping == Stepping::Single;
    }
    if (kernel == BDG_KERNEL_AUTO && sw.auto_pair && f.pair_usable && n_cols < 5) {
        reached.narrow_pair += small && p.stepping == Stepping::Pair;
        reached.narrow_single += !small && p.stepping == Stepping::Single;
    }

    // format: a kernel asked for by name keeps its format; the others take the best the copies allow
    int format = kernel;
    if (kernel == BDG_KERNEL_AUTO || kernel == BDG_KERNEL_AUTO_MOMENTS || kernel == BDG_KERNEL_PAIR || kernel == BDG_KERNEL_T2)
        format = f.diag_usable ? BDG_KERNEL_DICT_DIAG : f.dict_usable ? BDG_KERNEL_DICT : f.ell_usable ? BDG_KERNEL_ELL : BDG_KERNEL_DMMA;
    if (p.format != format) fail("format", kernel, n_cols, f, sw, p);
    if ((p.format == BDG_KERNEL_DICT_DIAG && !f.diag_usable) || (p.format == BDG_KERNEL_DICT && !f.dict_usable) ||
        (p.format == BDG_KERNEL_ELL && !f.ell_usable))
        fail("format without its flag", kernel, n_cols, f, sw, p);
    if (p.stepping != Stepping::Single && p.format != BDG_KERNEL_DICT && p.format != BDG_KERNEL_DICT_DIAG)
        fail("two-step plan off the dictionary", kernel, n_cols, f, sw, p);

    // panels
    const int width = p.stepping == Stepping::EvenCube ? 4 : p.stepping != Stepping::Single ? 8 : n_cols >= 5 ? 8 : n_cols >= 3 ? 4 : n_cols;
    if (p.panel_width != width) fail("panel width", kernel, n_cols, f, sw, p);
    if (!((long)p.n_panels * p.panel_width >= n_cols && n_cols > (long)(p.n_panels - 1) * p.panel_width))
        fail("panels do not cover the columns", kernel, n_cols, f, sw, p);
}

struct Pinned {
    const char *system;
    int kernel;
    PlanFacts facts;
    Stepping stepping;
    int format, panel_width, n_panels;
};

int main() {
    // the switches as bdg_cheb_begin reads them with none set
    for (const char *v : {"BDG_AUTO_PAIR", "BDG_AUTO_CUBE", "BDG_ELL_SD", "BDG_ELL_WALK", "BDG_ELL_PZ", "BDG_ELL_SEG", "BDG_ELL_PREFETCH",
                          "BDG_PAIR_SELF", "BDG_PAIR_OPEN", "BDG_PAIR_P", "BDG_PAIR_SEG", "BDG_PAIR_BALANCE", "BDG_CUBE_SHAPE",
                          "BDG_CUBE_SEG", "BDG_CUBE_BALANCE"})
        unsetenv(v);
    const PlanSwitches defaults = read_plan_switches();
    if (!defaults.auto_pair || !defaults.auto_cube) {
        std::printf("FAIL default switches: auto_pair=%d auto_cube=%d\n", defaults.auto_pair, defaults.auto_cube);
        return 1;
    }

    long plans = 0;
    const int kernels[] = {BDG_KERNEL_AUTO, BDG_KERNEL_DMMA, BDG_KERNEL_FMA, BDG_KERNEL_ELL, BDG_KERNEL_DICT,
                           BDG_KERNEL_DICT_DIAG, BDG_KERNEL_PAIR, BDG_KERNEL_T2, BDG_KERNEL_AUTO_MOMENTS};
    // Ly x Lz: (80, 88), (24, 296) and (88, 88) give 110, 111 and 121 patches of 8 x 8 per 4-column panel: below, at and above
    // 3/4 of 148 SMs with <= 4 columns
    const int sections[][2] = {{1, 1}, {100, 1}, {1000, 1}, {8, 8}, {64, 64}, {80, 88}, {24, 296}, {88, 88}, {200, 200}};
    for (int bits = 0; bits < 32; ++bits) {
        const bool ell = bits & 1, dict = bits & 2, diag = bits & 4, pair = bits & 8, cube = bits & 16;
        if ((diag && !dict) || (dict && !ell) || (pair && !dict) || (cube && !dict)) continue;  // diag => dict => ell; pair, cube => dict
        for (const long long n_sites : {4096LL, 65536LL, 65537LL, 1000000LL})
            for (const auto &yz : sections)
                for (int kernel : kernels)
                    for (int n_cols : {1, 2, 3, 4, 5, 8, 13, 41})
                        for (int sw_bits = 0; sw_bits < 4; ++sw_bits) {
                            PlanSwitches sw = defaults;
                            sw.auto_pair = sw_bits & 1;
                            sw.auto_cube = sw_bits & 2;
                            check(kernel, n_cols, PlanFacts{ell, dict, diag, pair, cube, n_sites, yz[0], yz[1], 148}, sw);
                            ++plans;
                        }
    }
    // A request that needs no copies (DMMA, FMA) plans from zero facts.
    for (int kernel : {BDG_KERNEL_DMMA, BDG_KERNEL_FMA})
        for (int n_cols : {1, 2, 3, 4, 5, 8, 13, 41}) {
            const SteppingPlan p = plan_stepping(kernel, n_cols, PlanFacts{}, defaults);
            if (p.refusal || p.stepping != Stepping::Single || p.format != kernel) fail("BSR plan", kernel, n_cols, PlanFacts{}, defaults, p);
        }
    if (!reached.refused || !reached.named || !reached.even_plane || !reached.even_cube || !reached.declined || !reached.narrow_pair ||
        !reached.narrow_single) {
        std::printf("FAIL coverage: refused %ld, named %ld, even plane %ld, cube %ld, declined %ld, narrow pair %ld, single %ld\n",
                    reached.refused, reached.named, reached.even_plane, reached.even_cube, reached.declined, reached.narrow_pair,
                    reached.narrow_single);
        return 1;
    }

    // The bench systems at 148 SMs, 8 columns, default switches: the facts ell_build finds for them and the plans they run on.
    //   C3: 100 x 100 x 1, d-wave + Rashba (complex hopping blocks: no diagonal dictionary)
    //   C4: 64 x 64 x 64, s-wave (two-dimensional x-planes: no pair kernel; open, real-diagonal hopping: the cube kernel)
    //   C5: 1000 x 1000 x 1 Josephson junction (real-diagonal hopping blocks)
    const PlanFacts c3{true, true, false, true, false, 10000, 100, 1, 148};
    const PlanFacts c4{true, true, true, false, true, 262144, 64, 64, 148};
    const PlanFacts c5{true, true, true, true, false, 1000000, 1000, 1, 148};
    const Pinned pinned[] = {
        {"C3", BDG_KERNEL_AUTO_MOMENTS, c3, Stepping::EvenPlane, BDG_KERNEL_DICT, 8, 1},
        {"C3", BDG_KERNEL_AUTO, c3, Stepping::Pair, BDG_KERNEL_DICT, 8, 1},
        {"C4", BDG_KERNEL_AUTO_MOMENTS, c4, Stepping::EvenCube, BDG_KERNEL_DICT_DIAG, 4, 2},
        {"C4", BDG_KERNEL_AUTO, c4, Stepping::Single, BDG_KERNEL_DICT_DIAG, 8, 1},
        {"C5", BDG_KERNEL_AUTO_MOMENTS, c5, Stepping::EvenPlane, BDG_KERNEL_DICT_DIAG, 8, 1},
        {"C5", BDG_KERNEL_AUTO, c5, Stepping::Pair, BDG_KERNEL_DICT_DIAG, 8, 1},
    };
    for (const Pinned &c : pinned) {
        const SteppingPlan p = plan_stepping(c.kernel, 8, c.facts, defaults);
        if (p.refusal || p.stepping != c.stepping || p.format != c.format || p.panel_width != c.panel_width || p.n_panels != c.n_panels) {
            std::printf("FAIL %s kernel %d: wanted %s / %d\n", c.system, c.kernel, name(c.stepping), c.format);
            fail("bench plan", c.kernel, 8, c.facts, defaults, p);
        }
    }
    std::printf("ok %ld plans, %ld refused\n", plans, reached.refused);
    return 0;
}
