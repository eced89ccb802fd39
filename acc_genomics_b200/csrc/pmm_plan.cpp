// pmm_plan.cpp -- see pmm_plan.h.
//
// What the reference does at this point is device-specific load balancing for its FPGA processing units
// (/root/reference/pairhmm/interface/PairHMMFpgaInterface.cpp:67-170) and tiling to the device limits
// (/root/reference/pairhmm/client/PairHMMWorker.cpp:217-221).  On the GPU there are no length limits; the
// planner's job is to keep lanes full (pick K x W per read length; wider lanes for jobs too small to fill the GPU), to
// make what a task pays once rare without lengthening the launch's tail (graded runs of haplotypes per task, longest
// first) and to keep the work queue deep enough for the 1 200 - 2 400 resident warps.
#include "pmm_plan.h"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <numeric>

namespace pmm {

// Maximise useful FP work per issue slot, 12*R / (W * step_cost(K)), subject to R + 1 <= K * W (one boundary row),
// with a mild penalty for variants whose register count lowers occupancy.
static Variant pick_variant_uncached(int R, int wmin);

Variant pick_variant(int R)
{
    // one answer per read length: looked up, not searched, for every read group of every job
    constexpr int kMemo = 1024;
    static const std::vector<Variant> memo = [] {
        std::vector<Variant> m(kMemo);
        for (int r = 0; r < kMemo; ++r) m[r] = pick_variant_uncached(r, 8);
        return m;
    }();
    return R >= 0 && R < kMemo ? memo[R] : pick_variant_uncached(R, 8);
}



// The same choice among the variants with at least wmin lanes per read (small jobs, see plan_job).
Variant pick_variant_wide(int R, int wmin)
{
    constexpr int kMemo = 1024;
    static const std::vector<Variant> memo16 = [] { std::vector<Variant> m(kMemo); for (int r = 0; r < kMemo; ++r) m[r] = pick_variant_uncached(r, 16); return m; }();
    static const std::vector<Variant> memo32 = [] { std::vector<Variant> m(kMemo); for (int r = 0; r < kMemo; ++r) m[r] = pick_variant_uncached(r, 32); return m; }();
    if (wmin <= 8) return pick_variant(R);
    if (R >= 0 && R < kMemo) return (wmin >= 32 ? memo32 : memo16)[R];
    return pick_variant_uncached(R, wmin);
}

static Variant pick_variant_uncached(int R, int wmin)
{
    Variant best{kStripedK, 32, true};
    double best_eff = -1.0;
    for (int W = wmin; W <= 32; W *= 2)
        for (int K = 4; K <= kMaxK; ++K) {
            if (!forward_f32_has_variant(K, W) || R + 1 > K * W) continue;
            double eff = 12.0 * R / (W * step_cost(K));
            if (K > 12) eff *= 0.97;
            if (eff > best_eff) { best_eff = eff; best = Variant{K, W, false}; }
        }
    return best;
}

struct Group { Variant v; uint32_t region; uint32_t reads[kMaxGroups]; uint32_t n; };

const PlanOptions& plan_defaults()
{
    static const PlanOptions d = [] {
        PlanOptions o;
        if (const char* e = std::getenv("PMM_SMALL_JOB_WIDENING"); e && *e) o.widening = std::atoi(e) != 0;
        if (const char* e = std::getenv("PMM_RUN_TIERS")) {
            int depth = kRunTierDepth, share = kRunTierShare, top = kRunTierTop;
            std::sscanf(e, "%d,%d,%d", &depth, &share, &top);
            o.tiers = RunTiers{std::max(0, std::min(64, depth)), std::max(1, std::min(100, share)), std::max(1, std::min(64, top))};
        }
        return o;
    }();
    return d;
}

// Every variant present costs one kernel launch, and a launch is inefficient when it has few tasks: it lasts at
// least as long as its longest task, and its tail leaves most of the GPU idle.  A mixed-length job (config 5: 10 % of
// the reads soft-clipped to 60..150 bases) picks eleven variants for 8 % of its work; measured on B200 for a 25-region
// job: every variant its own launch 3.37 ms, everything in the K = 19 launch 2.77 ms.  So: a variant moves up into the
// next larger one of the same W (same reads per warp, hence the same groups) whenever running its tasks with the
// unused rows is estimated cheaper than a launch of its own.  Smallest K first, so that moves cascade.
// Model (calibrated on that measurement): own launch = work / GPU rate + half the solo run time of the longest task
// (ramp + tail) + launch gap; moved = work at the larger variant's step cost / GPU rate.
static void merge_rare_variants(std::vector<Group>& groups, const std::vector<RegionDesc>& regions,
                                const uint32_t* hap_off, int sm_count, uint32_t longest_task_steps)
{
    constexpr double kSlotsPerUs = 1900.0;         // issue slots of one SMSP per microsecond (SM clock ~1.9 GHz)
    constexpr double kBusy = 0.85;                 // share of them this kernel uses on a full GPU
    constexpr double kSoloIpc = 0.55;              // what a warp alone on its SMSP reaches (dependent issue)
    constexpr double kLaunchUs = 4.0;              // launch gap
    double steps[3][kMaxK + 1] = {};               // [log2(W) - 3][K]: wavefront steps of all tasks of the variant
    auto widx = [](int W) { return W == 8 ? 0 : W == 16 ? 1 : 2; };
    for (const Group& g : groups) {
        if (g.v.striped) continue;
        const RegionDesc& r = regions[g.region];
        steps[widx(g.v.W)][g.v.K] += hap_off[r.hap_first + r.nhaps] - hap_off[r.hap_first] + r.nhaps;
    }
    const double gpu_slots_per_us = std::max(1, sm_count) * 4.0 * kSlotsPerUs * kBusy;
    int target[3][kMaxK + 1];
    bool any = false;
    for (int w = 0; w < 3; ++w) {
        for (int K = 0; K <= kMaxK; ++K) target[w][K] = K;
        for (int K = 1; K <= kMaxK; ++K) {
            if (steps[w][K] == 0) continue;
            int up = 0;
            for (int K2 = K + 1; K2 <= kMaxK && !up; ++K2) if (steps[w][K2] > 0) up = K2;
            if (!up) continue;
            const double own = steps[w][K] * step_cost(K) / gpu_slots_per_us +
                               0.5 * longest_task_steps * step_cost(K) / (kSlotsPerUs * kSoloIpc) + kLaunchUs;
            const double moved = steps[w][K] * step_cost(up) / gpu_slots_per_us;
            if (moved >= own) continue;
            steps[w][up] += steps[w][K];
            steps[w][K] = 0;
            target[w][K] = up; any = true;
        }
    }
    if (!any) return;
    for (Group& g : groups) {
        if (g.v.striped) continue;
        int K = g.v.K;
        const int w = widx(g.v.W);
        while (target[w][K] != K) K = target[w][K];
        g.v.K = K;
    }
}

int plan_job(uint32_t num_read, const uint32_t* read_off, uint32_t num_hap, const uint32_t* hap_off,
             uint32_t num_region, const pmm_region_t* regions, int sm_count, const PlanOptions& opt,
             Plan& plan, std::string& err, const std::function<Task*(const Plan&)>& task_dst)
{
    plan = Plan();
    const Variant* force = opt.force.K > 0 ? &opt.force : nullptr;
    if (!num_read || !num_hap || !num_region || !read_off || !hap_off || !regions) { err = "empty job"; return PMM_ERR_INVALID; }
    const uint64_t total_bases = (uint64_t)read_off[num_read] - read_off[0];
    const uint64_t total_hap = (uint64_t)hap_off[num_hap] - hap_off[0];
    if (read_off[num_read] < read_off[0] || hap_off[num_hap] < hap_off[0] || total_bases * 5 + total_hap >= (1ull << 31)) {
        err = "job larger than 2 GiB: split it"; return PMM_ERR_INVALID;
    }
    for (uint32_t i = 0; i < num_read; ++i) {
        if (read_off[i + 1] <= read_off[i]) { err = "read of length 0"; return PMM_ERR_INVALID; }
        plan.max_read_len = std::max(plan.max_read_len, read_off[i + 1] - read_off[i]);
    }
    for (uint32_t h = 0; h < num_hap; ++h) {
        if (hap_off[h + 1] <= hap_off[h]) { err = "haplotype of length 0"; return PMM_ERR_INVALID; }
        plan.max_hap_len = std::max(plan.max_hap_len, hap_off[h + 1] - hap_off[h]);
    }

    // ---- regions, result offsets, the reference's cell count (host/main.cpp:305-313) -------------------------
    plan.regions.resize(num_region);
    uint64_t rows = 0;
    for (uint32_t g = 0; g < num_region; ++g) {
        const pmm_region_t& r = regions[g];
        if (!r.num_read || !r.num_hap || (uint64_t)r.read_first + r.num_read > num_read ||
            (uint64_t)r.hap_first + r.num_hap > num_hap) { err = "region out of range"; return PMM_ERR_INVALID; }
        plan.regions[g] = RegionDesc{r.read_first, r.num_read, r.hap_first, r.num_hap, (uint32_t)plan.pairs, (uint32_t)rows};
        rows += r.num_read;
        plan.pairs += (uint64_t)r.num_read * r.num_hap;
        plan.cells += (uint64_t)(read_off[r.read_first + r.num_read] - read_off[r.read_first]) *
                      (uint64_t)(hap_off[r.hap_first + r.num_hap] - hap_off[r.hap_first]);
        if (plan.pairs >= (1ull << 31)) { err = "more than 2^31 pairs in one job: split it"; return PMM_ERR_INVALID; }
    }
    plan.rows = rows;

    // ---- small jobs: more lanes per read ---------------------------------------------------------------------------
    // The variant that wastes the fewest issue slots (151 bases: 19 rows x 8 lanes) makes long tasks -- a 450-base
    // haplotype is 110 000 instructions, ~90 us for a warp alone on its SMSP.  A job with fewer such tasks than the GPU has
    // SMSPs is over when its longest task is, so it is cut finer instead: with 16 or 32 lanes per read a task is a half
    // or a quarter as long and there are two or four times as many (a 10 x 5 toy region: float pass 85 -> ~30 us).  Wider
    // while the tasks still find at most two warps per SMSP.
    int wmin = 8;
    if (!force && opt.widening) {
        uint64_t t0 = 0;                                                // one-haplotype tasks with the default variants
        for (uint32_t g = 0; g < num_region; ++g) {
            const pmm_region_t& r = regions[g];
            double warps = 0;
            for (uint32_t k = 0; k < r.num_read; ++k) {
                const Variant v = pick_variant((int)(read_off[r.read_first + k + 1] - read_off[r.read_first + k]));
                warps += v.striped ? 1.0 : v.W / 32.0;
            }
            t0 += (uint64_t)(warps + 0.999) * r.num_hap;
        }
        const uint64_t two_per_smsp = (uint64_t)std::max(1, sm_count) * 8;
        wmin = t0 * 4 <= two_per_smsp ? 32 : t0 * 2 <= two_per_smsp ? 16 : 8;
    }

    // ---- read groups --------------------------------------------------------------------------------------------
    // Reads of a region are sorted by length (longest first); the longest unassigned read picks the (K, W)
    // variant and shares its warp with the next 32/W - 1 reads.
    std::vector<Group> groups;
    std::vector<uint32_t> order;
    uint64_t group_haps = 0, group_steps = 0;                          // summed over groups: haplotypes, wavefront steps
    for (uint32_t g = 0; g < num_region; ++g) {
        const pmm_region_t& r = regions[g];
        order.resize(r.num_read);
        std::iota(order.begin(), order.end(), r.read_first);
        std::stable_sort(order.begin(), order.end(), [&](uint32_t x, uint32_t y) {
            return read_off[x + 1] - read_off[x] > read_off[y + 1] - read_off[y]; });
        for (uint32_t k = 0; k < r.num_read;) {
            const int R = (int)(read_off[order[k] + 1] - read_off[order[k]]);
            Group gr; gr.region = g; gr.n = 0;
            gr.v = (force && !force->striped && forward_f32_has_variant(force->K, force->W) && R + 1 <= force->K * force->W)
                       ? *force : pick_variant_wide(R, wmin);
            const uint32_t G = gr.v.striped ? 1u : (uint32_t)(32 / gr.v.W);
            for (; gr.n < G && k < r.num_read; ++k) gr.reads[gr.n++] = order[k];
            for (uint32_t z = gr.n; z < (uint32_t)kMaxGroups; ++z) gr.reads[z] = 0;
            groups.push_back(gr);
            group_haps += r.num_hap;
            group_steps += hap_off[r.hap_first + r.num_hap] - hap_off[r.hap_first] + r.num_hap;
        }
    }

    // ---- runs of haplotypes: at least about tasks_per_warp queued tasks per resident warp (a bound that only jobs of more
    //      than ~38 000 group x haplotype units reach; below it the graded runs decide) --------------------------------
    const uint64_t resident_warps = (uint64_t)std::max(1, sm_count) * 16;
    const uint64_t target_tasks = std::max<uint64_t>(1, resident_warps * (uint64_t)std::max(1, opt.tasks_per_warp));
    plan.haps_per_task = (uint32_t)std::max<uint64_t>(1, (group_haps + target_tasks - 1) / target_tasks);
    // Graded runs.  What a task pays once -- its row-parameter loads and weight table, the wavefront's fill and drain, the
    // checked steps at both ends -- is about 3 % of a one-haplotype task, so long runs are cheaper; but the launch's tail is
    // as long as its last tasks.  Warps pull tasks longest first, so both are had by cutting a region's haplotypes into runs
    // of decreasing size: enough one-haplotype tasks for the last `depth` tasks of every resident warp, as many runs of
    // two before them, the rest in runs of `top` (ncu, config 2: 9.7 % of the float pass's warp samples lay outside the
    // steady loop with one haplotype per task).  A job with fewer than depth tasks per warp keeps one haplotype per task.
    double f1 = 0.0, f2 = 0.0;
    uint32_t top = plan.haps_per_task;
    const RunTiers& tiers = opt.tiers;
    if (tiers.depth > 0 && group_haps > 0) {
        // resident warps of the launch most groups belong to
        std::vector<uint32_t> by_k(kMaxK + 2, 0);
        for (const Group& g : groups) ++by_k[g.v.striped ? kMaxK + 1 : g.v.K];
        const int kmaj = (int)(std::max_element(by_k.begin(), by_k.end()) - by_k.begin());
        const uint64_t wr = (uint64_t)std::max(1, sm_count) * kWarpsPerCta * resident_ctas<float>(kmaj);
        const double u = (double)group_haps, u1 = (double)tiers.depth * wr, u2 = 2.0 * tiers.depth * wr;
        // the largest run: even made of the job's longest haplotypes, a task may not take more than `share` per cent of
        // the steps a warp does in the whole launch (config 4, 1-2 kb haplotypes and seven per warp: runs lose 5 %)
        const double warp_steps = (double)group_steps / wr;
        const uint32_t cap = (uint32_t)std::min<double>(tiers.top, warp_steps * tiers.share / 100.0 / (plan.max_hap_len + 1));
        if (cap >= 2) {
            f1 = std::min(1.0, u1 / u);
            f2 = cap == 2 ? 1.0 - f1 : std::min(1.0 - f1, u2 / u);
            top = std::max(top, cap);
        }
    }
    if (!force && !opt.keep_all_variants)
        merge_rare_variants(groups, plan.regions, hap_off, sm_count, top * (plan.max_hap_len + 1));

    // launches ordered by variant (largest footprint first); stable within a variant
    std::vector<uint32_t> gorder(groups.size());
    std::iota(gorder.begin(), gorder.end(), 0u);
    auto vkey = [](const Variant& v) { return (v.striped ? 1 << 20 : 0) + v.K * v.W * 64 + v.W; };
    std::stable_sort(gorder.begin(), gorder.end(), [&](uint32_t x, uint32_t y) { return vkey(groups[x].v) > vkey(groups[y].v); });

    // ---- runs of every region: all groups of a region walk the same cuts of its haplotypes, so the cuts, their costs
    //      (steps of the wavefront = haplotype bases + separators of the run) and, per launch, their cost classes are
    //      worked out once per region -- per task only a table lookup and one 48-byte store remain (16 000 tasks of
    //      config 2: 0.39 -> 0.1 ms of the host's staging time). mode 0: runs of haps_per_task, mode 1: one haplotype
    //      per task (striped reads) ------------------------------------------------------------------------------------
    struct RunTable { uint32_t first = 0, count = 0; };               // slice of run_h0 / run_cost (run_h0 has count + 1 entries)
    std::vector<RunTable> rt(2 * (size_t)num_region);
    std::vector<uint32_t> run_h0, run_cost;
    std::vector<uint8_t> run_cls;                                      // class of every run for the launch being laid out
    auto table_of = [&](uint32_t region, bool striped) -> const RunTable& {
        RunTable& t = rt[2 * (size_t)region + (striped ? 1 : 0)];
        if (t.count == 0) {
            const RegionDesc& r = plan.regions[region];
            const uint32_t* ho = hap_off + r.hap_first;
            // the region's haplotypes: `ones` runs of one at the end, `twos` runs of two before them, the rest in runs
            // of near-equal length of at most `top` (striped reads: one haplotype per task)
            const uint32_t n = r.nhaps;
            const uint32_t ones = striped ? n : std::min<uint32_t>(n, (uint32_t)(f1 * n + 0.5));
            const uint32_t twos = std::min<uint32_t>((n - ones) / 2, (uint32_t)(f2 * n / 2 + 0.5));
            const uint32_t rest = n - ones - 2 * twos;
            const uint32_t hpt = std::max(1u, std::min(top, rest));
            const uint32_t nrest = (rest + hpt - 1) / hpt;
            const uint32_t nruns = nrest + twos + ones;
            t.first = (uint32_t)run_h0.size(); t.count = nruns;
            for (uint32_t run = 0; run < nrest; ++run) run_h0.push_back((uint32_t)((uint64_t)rest * run / nrest));
            for (uint32_t run = 0; run < twos; ++run) run_h0.push_back(rest + 2 * run);
            for (uint32_t run = 0; run <= ones; ++run) run_h0.push_back(rest + 2 * twos + run);
            run_cost.resize(run_h0.size());
            for (uint32_t run = 0; run < nruns; ++run) {
                const uint32_t h0 = run_h0[t.first + run], h1 = run_h0[t.first + run + 1];
                run_cost[t.first + run] = ho[h1] - ho[h0] + (h1 - h0);
            }
        }
        return t;
    };

    // ---- pass A: group descriptors and launch segments -------------------------------------------------------------
    plan.groups.reserve(groups.size());
    uint64_t ntasks = 0;
    for (uint32_t gi : gorder) {
        const Group& gr = groups[gi];
        // row-parameter block of the group: every slot of the warp gets one, used or not
        GroupDesc gd{};
        for (uint32_t z = 0; z < (uint32_t)kMaxGroups; ++z) gd.read[z] = gr.reads[z];
        gd.nreads = gr.n; gd.K = (uint32_t)gr.v.K; gd.W = (uint32_t)gr.v.W;
        const uint32_t kw = gd.K * gd.W;
        gd.nstripes = gr.v.striped ? (read_off[gr.reads[0] + 1] - read_off[gr.reads[0]] + kw) / kw : 1u;
        const uint64_t slots = gr.v.striped ? 1u : 32u / gd.W;
        if (plan.param_floats + slots * gd.nstripes * kParamPlanes * kw >= (1ull << 32)) {
            err = "row parameters of one job exceed 16 GiB: split it"; return PMM_ERR_INVALID;
        }
        gd.param_off = (uint32_t)plan.param_floats;
        plan.param_floats += slots * gd.nstripes * kParamPlanes * kw;
        plan.groups.push_back(gd);
        if (plan.segs.empty() || !(plan.segs.back().v == gr.v)) plan.segs.push_back(LaunchSeg{gr.v, (uint32_t)ntasks, 0});
        const uint32_t nruns = table_of(gr.region, gr.v.striped).count;
        plan.segs.back().task_count += nruns;
        ntasks += nruns;
        if (ntasks >= (1ull << 31)) { err = "more than 2^31 warp-tasks in one job: split it"; return PMM_ERR_INVALID; }
    }
    plan.num_tasks = ntasks;

    // ---- where the tasks go: the caller's buffer (the engine's pinned staging arena) or plan.tasks ------------------
    Task* dst = nullptr;
    if (task_dst) {
        dst = task_dst(plan);
        if (!dst) { err = "no room for the task list"; return PMM_ERR_INVALID; }
    } else {
        plan.tasks.resize(ntasks);
        dst = plan.tasks.data();
    }

    // ---- pass B: write every task at its final position.  Longest tasks first inside each launch (warps pull tasks
    //      in order, so the kernel's tail is made of the shortest ones): a counting sort on 64 cost classes, stable,
    //      linear in the number of tasks, no intermediate copy. -----------------------------------------------------------
    run_cls.resize(run_cost.size());
    std::vector<uint32_t> regs_in_seg;                                  // regions met in the launch being laid out ...
    std::vector<uint32_t> groups_of(num_region, 0);                     // ... and how many of its groups each has
    size_t gk = 0;
    for (size_t sg = 0; sg < plan.segs.size(); ++sg) {
        const LaunchSeg& seg = plan.segs[sg];
        const bool striped = seg.v.striped;
        // the groups of this launch: gorder[gk .. gend)
        size_t gend = gk;
        uint32_t cmax = 1;
        regs_in_seg.clear();
        for (uint64_t tasks = 0; gend < gorder.size() && tasks < seg.task_count; ++gend) {
            const Group& gr = groups[gorder[gend]];
            const RunTable& t = table_of(gr.region, striped);
            if (groups_of[gr.region]++ == 0) {
                regs_in_seg.push_back(gr.region);
                for (uint32_t run = 0; run < t.count; ++run) cmax = std::max(cmax, run_cost[t.first + run]);
            }
            tasks += t.count;
        }
        uint32_t next[65] = {0};                                        // write cursor of each cost class
        for (uint32_t region : regs_in_seg) {
            const RunTable& t = table_of(region, striped);
            for (uint32_t run = 0; run < t.count; ++run) {
                const uint8_t cls = (uint8_t)(63 - (uint32_t)((uint64_t)run_cost[t.first + run] * 63 / cmax));
                run_cls[t.first + run] = cls;
                next[cls + 1] += groups_of[region];
            }
            groups_of[region] = 0;
        }
        next[0] = seg.task_first;
        for (int b = 0; b < 64; ++b) next[b + 1] += next[b];
        for (; gk < gend; ++gk) {
            const Group& gr = groups[gorder[gk]];
            const RegionDesc& r = plan.regions[gr.region];
            const GroupDesc& gd = plan.groups[gk];
            const RunTable& rtab = table_of(gr.region, striped);
            const uint32_t* h0s = run_h0.data() + rtab.first;
            const uint8_t* cls = run_cls.data() + rtab.first;
            Task proto;                                                  // everything of the task but its run
            for (uint32_t z = 0; z < (uint32_t)kMaxGroups; ++z) {
                proto.read[z] = gr.reads[z];
                proto.out_base[z] = z < gr.n ? r.out_first + (gr.reads[z] - r.read_first) * r.nhaps : 0;
            }
            proto.nreads = gr.n; proto.param_off = gd.param_off;
            for (uint32_t run = 0; run < rtab.count; ++run) {
                const uint32_t h0 = h0s[run], h1 = h0s[run + 1];
                Task& t = dst[next[cls[run]]++];
                t = proto;
                for (uint32_t z = 0; z < gr.n; ++z) t.out_base[z] += h0;
                t.hap_first = r.hap_first + h0; t.nhaps = h1 - h0;
            }
        }
    }
    return PMM_OK;
}

}  // namespace pmm
