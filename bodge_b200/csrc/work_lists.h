// Balanced plans of the two-applications-per-pass kernels (cheb_pair.cu, cheb_cube.cu): the (panel, patch column, x) space of
// a launch cut into one contiguous chunk per CTA slot and flattened into the device-side work lists the `LISTED` kernel
// instantiations read.  Host code, internal.
#pragma once

#include <algorithm>
#include <array>
#include <vector>

#include "bdg_internal.h"

namespace {

using WorkPiece = std::array<int, 4>;  // panel, patch column, x0, len

struct WorkPlan {
    std::vector<std::vector<WorkPiece>> per_cta;
    double longest = 0.0;  // iterations of the longest CTA: sum over its pieces of (len + piece_cost)
};

// `n_columns` patch columns of `Lx` planes per panel, `n_panels` panels, `slots` CTAs resident at a time.
// When a plane's columns fit the slots, CTAs come in groups of `n_columns` siblings -- one per column -- that march the SAME
// chunk of the (panel, x) space side by side: the halo sites a column needs from its neighbours are then in L2 when it reads
// them (as with the classic plan, which this reduces to for one panel), and every group gets an equal share of the planes.
// Otherwise (more columns than slots) the (panel, column, x) space is cut into one chunk per slot.
inline WorkPlan balanced_plan(int n_panels, int n_columns, int Lx, int64_t slots, int piece_cost, bool grouped) {
    WorkPlan plan;
    grouped = grouped && slots >= n_columns;
    const int64_t lanes = grouped ? slots / n_columns : slots;                     // chunks that run side by side
    const int64_t total = (int64_t)n_panels * (grouped ? 1 : n_columns) * Lx;      // plane units, panel(, column)-major
    const int64_t chunk = std::max<int64_t>(16, ceil_div(total, lanes));
    const int64_t n_chunks = ceil_div(total, chunk);
    int64_t begin = 0;
    for (int64_t c = 1; c <= n_chunks; ++c) {
        int64_t end = std::min(total, total * c / n_chunks);
        const int64_t into = end % Lx;  // a cut close to a column boundary moves onto it (no sliver pieces)
        if (c < n_chunks && into > 0 && into < 8) end -= into;
        else if (c < n_chunks && into > Lx - 8) end += Lx - into;
        if (end <= begin) continue;
        for (int col = 0; col < (grouped ? n_columns : 1); ++col) {
            std::vector<WorkPiece> mine;
            int64_t cost = 0;
            for (int64_t u = begin; u < end;) {
                const int64_t strip = u / Lx;  // grouped: the panel; else panel * n_columns + column
                const int x0 = (int)(u - strip * Lx), len = (int)std::min<int64_t>(Lx - x0, end - u);
                if (grouped) mine.push_back({(int)strip, col, x0, len});
                else mine.push_back({(int)(strip / n_columns), (int)(strip % n_columns), x0, len});
                cost += len + piece_cost;
                u += len;
            }
            plan.longest = std::max(plan.longest, (double)cost);
            plan.per_cta.push_back(std::move(mine));
        }
        begin = end;
    }
    return plan;
}

// The better of the two: siblings side by side, or one chunk of everything per slot -- whose halo reads miss L2 more often, so
// a kernel that runs close to the HBM roofline counts its length `flat_penalty` times (1.08 for the kernel of cheb_pair.cu;
// 1 for the shared-memory-bound one of cheb_cube.cu).
inline WorkPlan best_balanced_plan(int n_panels, int n_columns, int Lx, int64_t slots, int piece_cost, double flat_penalty) {
    WorkPlan grouped = balanced_plan(n_panels, n_columns, Lx, slots, piece_cost, true);
    if (slots < n_columns) return grouped;  // (that was the flat plan already)
    WorkPlan flat = balanced_plan(n_panels, n_columns, Lx, slots, piece_cost, false);
    flat.longest *= flat_penalty;
    return flat.longest < grouped.longest ? flat : grouped;
}

// Upload (WorkLists, bdg_internal.h: device pointers into `buf`): pieces (16-byte aligned: first), cta_begin[n_ctas + 1], run_panel[n_runs], panel_runs[n_panels + 1].  A run = a
// maximal sequence of pieces of one panel inside a CTA: its dot products go to partials[run].  Runs are numbered panel by
// panel (and in CTA order inside a panel), so the runs of panel p are panel_runs[p] .. panel_runs[p + 1] and the last one to
// arrive adds them up in that fixed order.
inline int upload_work_lists(bdg_system *sys, DevBuf &buf, const WorkPlan &plan, int n_panels, WorkLists &out) {
    struct Run { int panel, cta, order; };
    std::vector<Run> runs;
    std::vector<std::vector<int>> piece_run(plan.per_cta.size());
    for (size_t c = 0; c < plan.per_cta.size(); ++c) {
        int last_panel = -1;
        for (const WorkPiece &pc : plan.per_cta[c]) {
            if (pc[0] != last_panel) {
                last_panel = pc[0];
                runs.push_back({pc[0], (int)c, (int)runs.size()});
            }
            piece_run[c].push_back((int)runs.size() - 1);
        }
    }
    std::vector<Run> sorted = runs;
    std::stable_sort(sorted.begin(), sorted.end(), [](const Run &a, const Run &b) { return a.panel != b.panel ? a.panel < b.panel : a.cta < b.cta; });
    std::vector<int> id_of(runs.size()), run_panel(runs.size()), panel_runs(n_panels + 1, 0);
    for (size_t k = 0; k < sorted.size(); ++k) {
        id_of[sorted[k].order] = (int)k;
        run_panel[k] = sorted[k].panel;
        panel_runs[sorted[k].panel + 1] += 1;
    }
    for (int p = 0; p < n_panels; ++p) panel_runs[p + 1] += panel_runs[p];
    std::vector<int> flat, cta_begin{0};
    for (size_t c = 0; c < plan.per_cta.size(); ++c) {
        for (size_t k = 0; k < plan.per_cta[c].size(); ++k) {
            const WorkPiece &pc = plan.per_cta[c][k];
            flat.insert(flat.end(), {id_of[piece_run[c][k]], pc[1], pc[2], pc[3]});
        }
        cta_begin.push_back((int)(flat.size() / 4));
    }
    const size_t o_begin = flat.size(), o_rp = o_begin + cta_begin.size(), o_panel = o_rp + run_panel.size();
    flat.insert(flat.end(), cta_begin.begin(), cta_begin.end());
    flat.insert(flat.end(), run_panel.begin(), run_panel.end());
    flat.insert(flat.end(), panel_runs.begin(), panel_runs.end());
    BDG_TRY(dev_alloc(sys, buf, flat.size() * sizeof(int)));
    BDG_CUDA(cudaMemcpyAsync(buf.ptr, flat.data(), flat.size() * sizeof(int), cudaMemcpyHostToDevice, sys->stream));
    BDG_CUDA(cudaStreamSynchronize(sys->stream));  // `flat` goes out of scope
    const int *base = buf.as<int>();
    out.pieces = reinterpret_cast<const int4 *>(base);
    out.cta_begin = base + o_begin;
    out.run_panel = base + o_rp;
    out.panel_runs = base + o_panel;
    out.n_ctas = (int)plan.per_cta.size();
    out.n_runs = (int)runs.size();
    return BDG_OK;
}

// Classic or balanced plan for a launch of `n_items` items (patch, segment of `seg_len` planes) per panel on `slots` CTA slots.
// Classic: every panel has its own gx CTAs (grid = (gx, panels)), CTA (bx, panel) takes the items bx, bx + gx, ... (segment-
// major: the grid sweeps the lattice as one wavefront, so the halo sites of a patch are in L2 when its neighbour reads them);
// the kernel computes its items from the item index.  Balanced (best_balanced_plan): the (panel, patch, x) space cut into one
// contiguous chunk per CTA slot, handed to the kernel as lists -- no wave quantisation, no per-panel slot quantisation, fewer
// segment halos.  Taken when its longest CTA is clearly shorter (small lattices with many panels: C2 / C3: +3 .. +17 %); on
// large lattices the classic plan is near-perfect already.  `force`: 0 = classic, 1 = balanced, < 0 = decide.  `out`: the
// uploaded lists, or the classic plan's n_ctas = gx, n_runs = gx x panels and no lists.
inline int choose_work_plan(bdg_system *sys, DevBuf &buf, int n_panels, int n_patches, int Lx, int seg_len, int n_items,
                            int64_t slots, int piece_cost, double flat_penalty, int force, WorkLists &out) {
    const int gx = (int)std::min<int64_t>(std::max<int64_t>(1, slots / n_panels), n_items);
    const double classic_cost = (double)ceil_div((int64_t)gx * n_panels, slots) * (double)ceil_div(n_items, gx) * (seg_len + piece_cost);
    out = WorkLists();
    out.n_ctas = gx, out.n_runs = gx * n_panels;
    const WorkPlan plan = best_balanced_plan(n_panels, n_patches, Lx, slots, piece_cost, flat_penalty);
    if (!(force >= 0 ? force != 0 : plan.longest < 0.93 * classic_cost)) return BDG_OK;
    return upload_work_lists(sys, buf, plan, n_panels, out);
}

}  // namespace
