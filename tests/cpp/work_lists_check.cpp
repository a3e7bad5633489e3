// Host-side check of the balanced planner (bodge_b200/csrc/work_lists.h), built and run by tests/test_work_lists.py:
// every (panel, patch column, plane) unit is covered exactly once, pieces stay inside their column, the plan fits the CTA
// slots, and `longest` is the cost of the longest CTA.  Then the classic-or-balanced choice (choose_work_plan): forced
// either way, decided on either side of its threshold, and the lists it uploads.  No device code runs.
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "work_lists.h"

// Host stand-ins for what the upload calls: the lists land in host memory, where the checks read them.
int dev_alloc(bdg_system *, DevBuf &buf, size_t bytes) {
    buf.ptr = std::realloc(buf.ptr, bytes);
    buf.bytes = bytes;
    return buf.ptr ? BDG_OK : BDG_E_CUDA;
}
void bdg_set_error(const char *, ...) {}
extern "C" cudaError_t cudaMemcpyAsync(void *dst, const void *src, size_t count, cudaMemcpyKind, cudaStream_t) {
    std::memcpy(dst, src, count);
    return cudaSuccess;
}
extern "C" cudaError_t cudaStreamSynchronize(cudaStream_t) { return cudaSuccess; }
extern "C" const char *cudaGetErrorString(cudaError_t) { return "host stand-in"; }

struct Choice {
    int rc;
    WorkLists lists;
    double ratio;  // longest CTA of the best balanced plan / the classic plan's cost
};

static Choice choose(int n_panels, int n_patches, int Lx, int seg_len, long slots, int force) {
    static bdg_system sys;
    const int n_items = n_patches * (int)ceil_div(Lx, seg_len);
    Choice c{};
    c.rc = choose_work_plan(&sys, sys.cheb.work_items, n_panels, n_patches, Lx, seg_len, n_items, slots, 6, 1.08, force, c.lists);
    const int gx = (int)std::min<long>(std::max<long>(1, slots / n_panels), n_items);
    const double classic = (double)ceil_div((long)gx * n_panels, slots) * (double)ceil_div(n_items, gx) * (seg_len + 6);
    c.ratio = best_balanced_plan(n_panels, n_patches, Lx, slots, 6, 1.08).longest / classic;
    return c;
}

// The classic plan: no lists, gx CTAs per panel.
static bool is_classic(const Choice &c, int n_panels, int n_items, long slots) {
    const int gx = (int)std::min<long>(std::max<long>(1, slots / n_panels), n_items);
    return c.rc == BDG_OK && !c.lists.pieces && c.lists.n_ctas == gx && c.lists.n_runs == gx * n_panels;
}

// The uploaded lists hold the best balanced plan: the same pieces per CTA, runs numbered panel by panel.
static bool is_balanced(const Choice &c, int n_panels, int n_patches, int Lx, long slots) {
    const WorkPlan plan = best_balanced_plan(n_panels, n_patches, Lx, slots, 6, 1.08);
    const WorkLists &w = c.lists;
    if (c.rc != BDG_OK || !w.pieces || w.n_ctas != (int)plan.per_cta.size() || w.cta_begin[0] != 0) return false;
    if (w.panel_runs[0] != 0 || w.panel_runs[n_panels] != w.n_runs) return false;
    for (int cta = 0; cta < w.n_ctas; ++cta) {
        const std::vector<WorkPiece> &mine = plan.per_cta[cta];
        if (w.cta_begin[cta + 1] - w.cta_begin[cta] != (int)mine.size()) return false;
        for (size_t k = 0; k < mine.size(); ++k) {
            const int4 pc = w.pieces[w.cta_begin[cta] + k];
            if (pc.x < 0 || pc.x >= w.n_runs || w.run_panel[pc.x] != mine[k][0]) return false;
            if (pc.x < w.panel_runs[mine[k][0]] || pc.x >= w.panel_runs[mine[k][0] + 1]) return false;
            if (pc.y != mine[k][1] || pc.z != mine[k][2] || pc.w != mine[k][3]) return false;
        }
    }
    return true;
}

static int check(int n_panels, int n_columns, int Lx, long slots, int piece_cost, bool grouped_wanted) {
    const WorkPlan plan = balanced_plan(n_panels, n_columns, Lx, slots, piece_cost, grouped_wanted);
    std::vector<int> seen((size_t)n_panels * n_columns * Lx, 0);
    double longest = 0.0;
    if ((long)plan.per_cta.size() > slots || plan.per_cta.empty()) return 1;
    for (const auto &cta : plan.per_cta) {
        if (cta.empty()) return 2;
        double cost = 0.0;
        for (size_t k = 0; k < cta.size(); ++k) {
            const WorkPiece &pc = cta[k];
            if (pc[0] < 0 || pc[0] >= n_panels || pc[1] < 0 || pc[1] >= n_columns) return 3;
            if (pc[3] < 1 || pc[2] < 0 || pc[2] + pc[3] > Lx) return 4;
            // a CTA walks the space in ascending (panel, column, x) order: its dot-product runs are contiguous per panel
            if (k && (pc[0] < cta[k - 1][0])) return 5;
            for (int x = pc[2]; x < pc[2] + pc[3]; ++x) seen[((size_t)pc[0] * n_columns + pc[1]) * Lx + x] += 1;
            cost += pc[3] + piece_cost;
        }
        if (cost > longest) longest = cost;
    }
    for (int v : seen)
        if (v != 1) return 6;
    if (longest != plan.longest) return 7;
    return 0;
}

int main() {
    long cases = 0;
    for (int n_panels : {1, 2, 3, 7, 32, 64, 512})
        for (int n_columns : {1, 2, 7, 8, 9, 72, 300})
            for (int Lx : {3, 4, 7, 8, 9, 15, 16, 17, 64, 100, 250, 1000})
                for (long slots : {1L, 2L, 7L, 148L, 296L, 444L})
                    for (int piece_cost : {0, 5})
                        for (int grouped = 0; grouped < 2; ++grouped) {
                            if ((long)n_panels * n_columns * Lx > 2000000L) continue;  // keep the run to seconds
                            const int rc = check(n_panels, n_columns, Lx, slots, piece_cost, grouped != 0);
                            if (rc) {
                                std::printf("FAIL rc=%d panels=%d columns=%d Lx=%d slots=%ld cost=%d grouped=%d\n", rc, n_panels,
                                            n_columns, Lx, slots, piece_cost, grouped);
                                return 1;
                            }
                            ++cases;
                        }
    // the better-of-two choice never returns a plan longer than the grouped one
    for (int n_panels : {1, 8, 64})
        for (int n_columns : {7, 8, 72}) {
            const WorkPlan best = best_balanced_plan(n_panels, n_columns, 100, 296, 5, 1.08);
            const WorkPlan grouped = balanced_plan(n_panels, n_columns, 100, 296, 5, true);
            if (best.longest > grouped.longest) {
                std::printf("FAIL best plan longer than the grouped one: panels=%d columns=%d\n", n_panels, n_columns);
                return 1;
            }
        }
    // classic or balanced: forced either way, else the balanced plan when its longest CTA is < 0.93 of the classic cost
    int below = 0, above = 0;
    for (int n_panels : {1, 2, 8, 64})
        for (int n_patches : {1, 7, 72})
            for (int Lx : {16, 100, 1000})
                for (int seg_len : {4, 16, 100})
                    for (long slots : {148L, 296L}) {
                        if (seg_len > Lx) continue;
                        const int n_items = n_patches * (int)ceil_div(Lx, seg_len);
                        const Choice classic = choose(n_panels, n_patches, Lx, seg_len, slots, 0);
                        const Choice balanced = choose(n_panels, n_patches, Lx, seg_len, slots, 1);
                        const Choice decided = choose(n_panels, n_patches, Lx, seg_len, slots, -1);
                        const bool want = decided.ratio < 0.93;
                        if (!is_classic(classic, n_panels, n_items, slots) || !is_balanced(balanced, n_panels, n_patches, Lx, slots) ||
                            !(want ? is_balanced(decided, n_panels, n_patches, Lx, slots) : is_classic(decided, n_panels, n_items, slots))) {
                            std::printf("FAIL choice: panels=%d patches=%d Lx=%d seg=%d slots=%ld ratio=%.4f\n", n_panels, n_patches, Lx,
                                        seg_len, slots, decided.ratio);
                            return 1;
                        }
                        below += decided.ratio >= 0.85 && want;
                        above += !want && decided.ratio < 1.0;
                    }
    if (!below || !above) {  // the sweep must reach both sides of the threshold close to it
        std::printf("FAIL choice: %d plans in [0.85, 0.93), %d in [0.93, 1)\n", below, above);
        return 1;
    }
    std::printf("ok %ld plans, choice %d + %d near the threshold\n", cases, below, above);
    return 0;
}
