/*
 * pairhmm_cuda.h -- C ABI of the B200 PairHMM forward engine (libpairhmm_b200.so).
 *
 * This is the thin layer that replaces the reference's FPGA/OpenCL dispatch for the PairHMM path.  Plain C,
 * plain pointers and sizes, integer status codes, no exceptions across the boundary, caller-owned output
 * buffers.  Every entry point names the reference interface it stands in for (paths under
 * /root/reference/pairhmm/).  INTEGRATION.md shows the bindings a maintainer of the reference would add.
 *
 * Semantics common to all compute calls
 *   - A "region" is a cross product: num_read reads against num_hap haplotypes; results are read-major,
 *     out[i * num_hap + j] for read i and haplotype j (host/main.cpp:365, client/PairHMMWorker.cpp:171-193).
 *   - "raw" results are the float likelihoods scaled by 2^120 that the reference's accelerators return in the
 *     task's output block (task/xlnx/PairHMMTask.cpp:69-79) and that compute_fp_avxs returns on the CPU
 *     (xlnx/host/avx_impl.cpp:4); they are bit-identical to the AVX implementation built without FMA contraction.
 *   - "log10" results are the final doubles of PairHMMWorker::getOutput (client/PairHMMWorker.cpp:157-197):
 *     raw < 1e-28f selects the double-precision re-run, log10(d) - log10(2^1020); otherwise
 *     (double)(log10f(raw) - log10f(2^120)).  The re-run happens on the GPU; log10 is taken with the host libm.
 *   - Quality bytes are used modulo 128 and any base other than A,C,G,T,N counts as A, like the reference
 *     (xlnx/host/avx-pairhmm-template.h:110-112, xlnx/host/host_type.h:123-143).  Reads and haplotypes of length 0
 *     are rejected with PMM_ERR_INVALID (the reference reads uninitialised memory for them).
 *   - A pmm_ctx is bound to one GPU and is not thread-safe; use one context per host thread (as the reference
 *     uses one PairHMMClient per thread).  Different contexts may be used concurrently.
 */
#ifndef PAIRHMM_CUDA_H
#define PAIRHMM_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct pmm_ctx pmm_ctx;

enum {
    PMM_OK = 0,
    PMM_ERR_INVALID = 1,     /* bad argument / malformed buffer                     */
    PMM_ERR_CUDA = 2,        /* CUDA runtime error, text in pmm_last_error()        */
    PMM_ERR_NO_DEVICE = 3,   /* no usable GPU: the engine has NO CPU fallback       */
    PMM_ERR_STATE = 4        /* call sequence violated (e.g. fetch before launch)   */
};

/* Same field order and meaning as read_t / hap_t (interface/PairHMMHostInterface.h:27-39). */
typedef struct { int len; char* _b; char* _q; char* _i; char* _d; char* _c; } pmm_read_t;
typedef struct { int len; char* _b; } pmm_hap_t;

/* One region of a flat multi-region job: reads [read_first, +num_read) x haplotypes [hap_first, +num_hap). */
typedef struct { uint32_t read_first, num_read, hap_first, num_hap; } pmm_region_t;

typedef struct {
    uint64_t pairs, cells;            /* cells = sum over regions of sum(read_len) * sum(hap_len) (host/main.cpp:305-313) */
    uint64_t fallback_pairs;          /* pairs re-run in double (raw < 1e-28f)                              */
    uint64_t flush_pairs;             /* of those, re-run again with x86 flush-to-zero emulation             */
    uint64_t h2d_bytes, d2h_bytes;
    uint32_t kernel_launches;         /* kernels launched by the last pmm_launch                             */
    uint32_t f32_tasks;               /* warp-tasks of the float pass                                        */
    float    ms_stage, ms_f32, ms_fallback, ms_fetch;   /* CUDA-event / host timings of the last job          */
    uint64_t recheck_pairs;           /* fast mode: pairs re-run by the exact float kernel (guard band)      */
} pmm_stats_t;

/* ---- lifetime ------------------------------------------------------------------------------------------
 * Replaces: lazy `new OpenCLEnv(bit_path, KERNEL_NAME)` in compute_fpga (host/PairHMMFpga.cpp:131-133) and the
 * Blaze TaskEnv the task obtains with getEnv() (task/xlnx/PairHMMTask.cpp:30).  device < 0 picks the current one. */
int  pmm_create(int device, pmm_ctx** out);
void pmm_destroy(pmm_ctx* ctx);
const char* pmm_last_error(const pmm_ctx* ctx);     /* ctx may be NULL: last error of pmm_create */
int  pmm_device_count(void);

/* Options (strings, like the task's get_conf(key, value), task/xlnx/PairHMMTask.h:73-77):
 *   "stream"          = value of a cudaStream_t (decimal or 0x..) to run on, "default" for the legacy default
 *                       stream, "own" for the context's own non-blocking stream (the initial setting)
 *   "priority"        = rank of this context among the contexts that share its GPU, 0 = first in line (the highest CUDA
 *                       stream priority), larger = later; replaces the context's own stream.  Decides whose thread blocks take
 *                       the SM slots another context's kernel frees at its tail
 *   "tasks_per_warp"  = target queue depth per resident warp used when cutting regions into warp-tasks
 *   "small_job_widening" = "on" (default): a job with fewer warp-tasks than the GPU can spread over its SMSPs gets 16 or 32
 *                       lanes per read instead of the variant that wastes the fewest issue slots -- shorter, more numerous
 *                       tasks, i.e. a shorter critical path for a per-region caller.  For this context
 *   "run_tiers"       = "depth[,share[,top]]", graded runs: a region's haplotypes are cut into runs of decreasing size (long
 *                       runs first, so what a task pays once is paid rarely; one-haplotype tasks last, so the launch's tail
 *                       stays short): `depth` tasks per resident warp in each tier (default 2; 0 = runs of equal size), no
 *                       task longer than `share` per cent of a warp's steps in the launch (40), at most `top` haplotypes
 *                       per run (4).  For this context
 *   "mode"            = "exact" (default): every multiply and add of the float pass is rounded on its own, results are
 *                       bit-identical to the reference's AVX code.  "fast": the float cell update is contracted to
 *                       4 FMUL + 4 FFMA per cell (12 -> 8 instructions); results agree with the reference to a few
 *                       float ulp (<= 1e-5 relative in log10, typically 1e-7), and every pair whose float result lies
 *                       within the guard band around 1e-28f is re-run by the exact kernel before the float-versus-
 *                       double decision is taken, so that decision stays identical to the reference's
 *   "guard"           = relative half-width of that band (default 0.0078125 = 2^-7)
 *   "force_variant"   = "K,W": rows per lane and lanes per read of the float kernel for every read that fits
 *                       (tuning sweeps, tools/sweep_variants.py); "0,0" gives the choice back to the planner,
 *                       "-1,0" keeps every variant in a launch of its own (no consolidation of rare ones)
 *   "f64_tasks_per_warp", "f64_max_run" = how the double re-run cuts a read's failing haplotypes into tasks: about
 *                       f64_tasks_per_warp tasks per resident warp (default 6), at most f64_max_run haplotypes each (6)
 *   "overlap"         = "on" (default): the launch stream waits, after a launch, for the double re-run of the launch BEFORE, so
 *                       consecutive launches overlap by one pass; "off": for its own re-run, every launch is complete on
 *                       the launch stream when the next thing queued there starts (what per-launch event brackets need)
 *   "sync"            = "spin" (default): waits poll the stream, lowest latency for one context per core; "block":
 *                       waits sleep on a blocking event (for hosts with fewer cores than waiting threads); "hybrid": poll
 *                       for 60 us, then sleep; "auto": spin while fewer than cores/16 threads of the process do, else sleep.  The pool takes it from the environment variable PMM_POOL_SYNC, the task
 *                       plugin from its conf key "sync" or PAIRHMM_SYNC                                              */
int  pmm_set_option(pmm_ctx* ctx, const char* key, const char* value);

/* ---- one-shot calls, host buffers in, host buffers out --------------------------------------------------
 * pmm_forward_raw_serialized replaces PairHMM::prepare() + PairHMM::compute() (task/xlnx/PairHMMTask.cpp:27-143)
 * and compute_fpga (host/PairHMMFpga.h:16-20): inputs are the task's input blocks 1 and 2 -- the byte streams of
 * serialize() (interface/PairHMMHostInterface.cpp:175-207) -- and the output is the task's output block 0.
 * out_raw must hold num_read * num_hap floats; the counts are returned through num_read / num_hap. */
int  pmm_forward_raw_serialized(pmm_ctx* ctx, const void* reads_ser, uint64_t reads_bytes,
                                const void* haps_ser, uint64_t haps_bytes,
                                float* out_raw, uint64_t out_capacity, int* num_read, int* num_hap);

/* Replaces PairHMMWorker::run() + getOutput() (client/PairHMMWorker.cpp:157-271) and
 * FalconPairHMM::computePairhmmAVX (xlnx/host/FalconPairHMM.cpp:69-95) for one region. */
int  pmm_forward_log10(pmm_ctx* ctx, const pmm_read_t* reads, int num_read, const pmm_hap_t* haps, int num_hap,
                       double* out, uint64_t* n_fallback);
int  pmm_forward_log10_serialized(pmm_ctx* ctx, const void* reads_ser, uint64_t reads_bytes,
                                  const void* haps_ser, uint64_t haps_bytes,
                                  double* out, uint64_t out_capacity, int* num_read, int* num_hap,
                                  uint64_t* n_fallback);

/* The GKL-shaped batch entry (what Intel GKL's JNI computeLikelihoods builds and what the reference's worker converts
 * its reads and haplotypes into, client/PairHMMWorker.cpp:113-127): one `testcase` per pair, same field order as
 * xlnx/host/host_type.h:69-73, read-major, the pointers of a read shared by the pairs of its row and the pointers of a
 * haplotype by the pairs of its column.  out[k] is the final log10 likelihood of tc[k] -- what the per-pair loop
 * compute_fp_avxs / compute_fp_avxd + log10 of FalconPairHMM::computePairhmmAVX (xlnx/host/FalconPairHMM.cpp:69-95)
 * returns.  Pairs that share a read (consecutive testcases with the same read pointers) are grouped into regions
 * internally; any sequence of testcases is accepted, a full cross product is simply the one-region case. */
typedef struct { int rslen, haplen; const char *q, *i, *d, *c; const char *hap, *rs; } pmm_testcase_t;
int  pmm_forward_log10_testcases(pmm_ctx* ctx, const pmm_testcase_t* tc, uint64_t n, double* out, uint64_t* n_fallback);

/* ---- staged calls: many regions per job, device-resident between steps -----------------------------------
 * The flat layout is five parallel byte arrays for the reads (bases, base / insertion / deletion /
 * gap-continuation qualities) indexed by read_off[0..num_read], one byte array for the haplotypes indexed by
 * hap_off[0..num_hap], and a list of regions.  Results of region g start at sum over earlier regions of
 * num_read * num_hap.
 *   pmm_stage_flat : pack into pinned memory, copy to the GPU, build the haplotype stream and the task queue
 *   pmm_launch     : float pass + fallback compaction + double re-run; asynchronous on the context's stream
 *   pmm_fetch_*    : wait, copy results back, (log10) finish on the host
 * pmm_launch may be called repeatedly on one staged job (bench.py times it with inputs resident in HBM); consecutive
 * launches overlap by one pass: the float pass of launch i + 1 runs beside the double re-run of launch i. */
int  pmm_stage_flat(pmm_ctx* ctx, uint32_t num_read, const uint32_t* read_off,
                    const uint8_t* bases, const uint8_t* q, const uint8_t* i, const uint8_t* d, const uint8_t* c,
                    uint32_t num_hap, const uint32_t* hap_off, const uint8_t* hap_bases,
                    uint32_t num_region, const pmm_region_t* regions);
/* Same, from the task's serialized input blocks (what PairHMM::prepare() receives, task/xlnx/PairHMMTask.cpp:35-38). */
int  pmm_stage_serialized(pmm_ctx* ctx, const void* reads_ser, uint64_t reads_bytes,
                          const void* haps_ser, uint64_t haps_bytes, int* num_read, int* num_hap);
int  pmm_launch(pmm_ctx* ctx);
/* The double re-run of a launch runs on a stream of its own, next to the float pass of the following launch; pmm_launch
 * itself only makes the launch stream wait for the re-run of the launch BEFORE.  pmm_join makes the launch stream wait
 * for the last launch's re-run too (no host wait): what a caller records on that stream afterwards -- an event closing
 * a timed region, say -- comes after all kernels of all launches so far. */
int  pmm_join(pmm_ctx* ctx);
int  pmm_sync(pmm_ctx* ctx);
int  pmm_fetch_raw(pmm_ctx* ctx, float* out_raw, uint64_t out_capacity);
int  pmm_fetch_log10(pmm_ctx* ctx, double* out, uint64_t out_capacity, uint64_t* n_fallback);
/* The pairs that took the double re-run: index[k] = position in the read-major result, value[k] = the double
 * likelihood scaled by 2^1020 (what compute_fp_avxd returns, client/PairHMMWorker.cpp:182).  With index == value ==
 * NULL only the count is returned. */
int  pmm_fetch_fallback(pmm_ctx* ctx, uint32_t* index, double* value, uint64_t capacity, uint64_t* count);
/* The fallback decision of the last launched job: mask[k] = 1 where raw[k] < 1e-28f. */
int  pmm_fetch_fallback_mask(pmm_ctx* ctx, uint8_t* mask, uint64_t capacity);

int  pmm_get_stats(const pmm_ctx* ctx, pmm_stats_t* out);

/* Where the kernels of the last launched job sit on the device's clock, for idle-time analysis of the work queue:
 * seconds since the context's reference event (recorded when the context was created), and the host's steady clock
 * (std::chrono::steady_clock, seconds) at that reference.  Waits for the job's kernels. */
typedef struct { double ref_host_s, kernels_start_s, f32_end_s, kernels_end_s; } pmm_timeline_t;
int  pmm_get_timeline(pmm_ctx* ctx, pmm_timeline_t* out);

/* ---- multi-GPU work queue --------------------------------------------------------------------------------
 * Independent read x haplotype regions are partitioned across the GPUs of one box by a host-side queue; nothing is
 * reduced, so there is no collective (SURVEY.md section 8e).  The pool owns contexts_per_device contexts on each of
 * the given devices (NULL / 0 = every visible GPU) and one feeder thread per pair of contexts of a device; each
 * submitted job runs as one GPU job, served by generation (a run of consecutive tickets) and largest first inside one.
 * This is what stands where the reference has Blaze's accelerator queue (client/PairHMMWorker.cpp:217-251 hands
 * tiles to client_->start() one after another) and the per-PU balancer (interface/PairHMMFpgaInterface.cpp:67-170).
 *   pmm_pool_submit_flat : same layout as pmm_stage_flat (regions == NULL: one region of everything); the input
 *                          arrays and out_log10 are borrowed until pmm_pool_wait(ticket) returns.  Thread-safe.
 *   pmm_pool_wait        : blocks until that job is done; returns the job's status, the number of pairs that took
 *                          the double re-run and the device that ran it.  Each ticket is waited for exactly once. */
typedef struct pmm_pool pmm_pool;
int  pmm_pool_create(const int* devices, int n_devices, int contexts_per_device, pmm_pool** out);
void pmm_pool_destroy(pmm_pool* pool);
const char* pmm_pool_last_error(const pmm_pool* pool);      /* pool may be NULL: last error of pmm_pool_create */
int  pmm_pool_num_devices(const pmm_pool* pool);
int  pmm_pool_submit_flat(pmm_pool* pool, uint32_t num_read, const uint32_t* read_off,
                          const uint8_t* bases, const uint8_t* q, const uint8_t* i, const uint8_t* d, const uint8_t* c,
                          uint32_t num_hap, const uint32_t* hap_off, const uint8_t* hap_bases,
                          uint32_t num_region, const pmm_region_t* regions,
                          double* out_log10, uint64_t out_capacity, uint64_t* ticket);
int  pmm_pool_wait(pmm_pool* pool, uint64_t ticket, uint64_t* n_fallback, int* device);
/* Jobs and cells completed so far by the slot-th device of the pool (0 <= slot < pmm_pool_num_devices). */
int  pmm_pool_device_load(const pmm_pool* pool, int slot, int* device, uint64_t* jobs, uint64_t* cells);
/* Timeline of the pool's GPU jobs (one record per submitted job that ran without error), for finding idle time:
 * host times of the feeder's stages and the device times of the job's kernels, all in seconds since the pool was
 * created.  pmm_pool_trace(pool, 1) starts recording (and clears), 0 stops; pmm_pool_get_trace copies up to capacity
 * records and returns how many exist. */
typedef struct {
    int32_t  device, context;           /* CUDA device and the pool's context index that ran the job          */
    uint32_t regions;                   /* regions in the job                                                   */
    uint64_t cells, pairs;
    double   t_take, t_staged, t_launched, t_fetched;   /* host: job taken from the queue, pmm_stage_flat returned,
                                                            pmm_launch returned, results delivered                */
    double   d_start, d_f32_end, d_end; /* device: first kernel starts, float pass ends, double re-run ends      */
} pmm_pool_trace_t;
int  pmm_pool_trace(pmm_pool* pool, int on);
int  pmm_pool_get_trace(pmm_pool* pool, pmm_pool_trace_t* out, uint64_t capacity, uint64_t* count);

/* ---- host-only entry points (no GPU needed) -------------------------------------------------------------
 * pmm_plan_flat: how pmm_stage_flat would cut a job into warp-tasks on a GPU with sm_count SMs.  This is the
 * planner that stands where the reference balances reads over FPGA processing units and tiles batches to
 * 2048 x 128 (interface/PairHMMFpgaInterface.cpp:67-170, client/PairHMMWorker.cpp:217-221).  With out == NULL
 * only the count is returned.  Errors are reported through pmm_last_error(NULL). */
typedef struct {
    uint32_t read[4];          /* reads sharing the warp (num_read of them are valid)                    */
    uint32_t out_base[4];      /* result index of (read[g], hap_first)                                    */
    uint32_t hap_first, num_hap, num_read;
    uint32_t rows_per_lane, lanes_per_read, striped;   /* kernel variant: K, W, multi-stripe flag         */
} pmm_task_info_t;
int  pmm_plan_flat(uint32_t num_read, const uint32_t* read_off, uint32_t num_hap, const uint32_t* hap_off,
                   uint32_t num_region, const pmm_region_t* regions, int sm_count, int tasks_per_warp,
                   pmm_task_info_t* out, uint64_t capacity, uint64_t* num_tasks);
/* The probability tables the engine uploads, as generated by the host libm following Context<NUMBER>
 * (xlnx/host/Context.h:42-61,:105-110,:145-151).  which: 0 ph2pr f32[128], 1 matchToMatch f32[8256],
 * 2 ph2pr f64[128], 3 matchToMatch f64[8256], 4 log10(2^120) f32, 5 log10(2^1020) f64. */
int  pmm_host_table(int which, void* out, uint64_t capacity_bytes);

/* The host-side tail of PairHMMWorker::getOutput (client/PairHMMWorker.cpp:157-197) for callers that hold the raw floats
 * and the fallback list (task output blocks 0 and 1): out[k] = (double)(log10f(raw[k]) - log10f(2^120)), then
 * out[fb_index[j]] = log10(fb_value[j]) - log10(2^1020).  Host libm, several threads. */
int  pmm_host_finish_log10(const float* raw, uint64_t n, const uint32_t* fb_index, const double* fb_value, uint64_t n_fb,
                           double* out);

/* Measured FP32 instruction issue rate of this GPU in lane-instructions per second (the roofline denominator of
 * SURVEY.md section 8d; an independent FMUL/FADD stream, ~20 ms).  Also returns the SM clock seen while measuring. */
int  pmm_measure_fp32_peak(pmm_ctx* ctx, double* lane_instr_per_s, double* sm_mhz);
/* The same for the FP64 pipe (independent DMUL/DADD streams): the denominator of the double re-run's roofline. */
int  pmm_measure_fp64_peak(pmm_ctx* ctx, double* lane_instr_per_s);

#ifdef __cplusplus
}
#endif
#endif /* PAIRHMM_CUDA_H */
