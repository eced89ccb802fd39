// pmm_plan.h -- host-side planner: cuts a job (regions of reads x haplotypes) into warp-tasks.  Pure C++, no CUDA,
// so that the CPU test-suite can check it (tests/test_plan.py through pmm_plan_flat).
#pragma once
#include <functional>
#include <string>
#include <vector>

#include "../../include/pairhmm_cuda.h"
#include "pmm_types.h"

namespace pmm {

struct LaunchSeg { Variant v; uint32_t task_first, task_count; };

struct Plan {
    std::vector<RegionDesc> regions;
    std::vector<GroupDesc> groups;      // read groups (reads sharing a warp) and where their row parameters live
    uint64_t param_floats = 0;          // size of the row-parameter buffer
    std::vector<Task> tasks;            // grouped by variant, see segs (empty when the caller supplied the destination)
    uint64_t num_tasks = 0;
    std::vector<LaunchSeg> segs;        // one kernel launch each, largest footprint first
    uint64_t pairs = 0, cells = 0, rows = 0;   // rows: result rows = reads summed over regions
    uint32_t max_hap_len = 0, max_read_len = 0;
    uint32_t haps_per_task = 0;
};

// Issue slots one step of K cells costs in the float kernel (from the SASS of the steady loop: 12 FP per cell,
// one LDS.128 per 4 rows, and 3 SHFL + LDG + 2 sum FADD + address/loop overhead per step).
inline double step_cost(int K) { return 12.25 * K + 9.0; }

// Graded runs (plan_job): `depth` tasks per resident warp in each tier of run sizes (0 = runs of equal size); no task
// longer than `share` per cent of a warp's steps in the launch; at most `top` haplotypes per run.
struct RunTiers { int depth, share, top; };
constexpr int kRunTierDepth = 2, kRunTierShare = 40, kRunTierTop = 4;

// How plan_job cuts a job.  Each engine context owns one (pmm_set_option); a new context and pmm_plan_flat start from
// plan_defaults().
struct PlanOptions {
    // Small jobs (fewer one-haplotype tasks than two warps per SMSP could take after widening) get more lanes per read,
    // i.e. shorter and more tasks.
    bool widening = true;
    RunTiers tiers{kRunTierDepth, kRunTierShare, kRunTierTop};
    int tasks_per_warp = 16;            // queue depth per resident warp
    Variant force{0, 0, false};         // tuning sweeps: K > 0 = this variant for every read that fits it
    bool keep_all_variants = false;     // tuning sweeps: every variant a launch of its own (no consolidation of rare ones)
};

// The defaults, with PMM_SMALL_JOB_WIDENING=0|1 and PMM_RUN_TIERS="depth[,share[,top]]" applied (read once per process).
const PlanOptions& plan_defaults();

// Best (K, W) for a read of R bases; pick_variant_wide: among the variants with at least wmin lanes per read.
Variant pick_variant(int R);
Variant pick_variant_wide(int R, int wmin);

// Returns PMM_OK or PMM_ERR_INVALID with a message.
int plan_job(uint32_t num_read, const uint32_t* read_off, uint32_t num_hap, const uint32_t* hap_off,
             uint32_t num_region, const pmm_region_t* regions, int sm_count, const PlanOptions& opt,
             Plan& plan, std::string& err,
             // called once the task count (plan.num_tasks), groups and launches are known; returns where to write the tasks
             const std::function<Task*(const Plan&)>& task_dst = nullptr);

}  // namespace pmm
