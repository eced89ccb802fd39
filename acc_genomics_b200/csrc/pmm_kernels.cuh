// pmm_kernels.cuh -- device-side data model of the B200 PairHMM forward engine (declarations shared by the
// kernels in pmm_kernels.cu and the C ABI in pmm_engine.cu).
//
// Layout in HBM (one "job" = any number of active regions, each a reads x haplotypes cross product):
//   read blob      bytes; per read five tracks (_b,_q,_i,_d,_c) found through ReadDesc{off, stride, len}: track t of
//                  read r is blob[off + t*stride .. +len).  stride = len for the reference's wire format
//                  (PairHMMHostInterface.cpp:175-192), stride = total bases for five flat arrays.
//   hap blob       bytes; HapDesc{off, len}.
//   hap stream     bytes; all haplotypes of the job back to back, each preceded by a separator:
//                  SEP c c c ... c SEP c c ... c SEP(final).  c = base class 0..4 (A,C,T,G,N; every other byte is
//                  class 0 exactly like ConvertChar, host_type.h:123-143).  hap h starts at stream[spos[h]] (its SEP).
//   initY          per hap, INITIAL_CONSTANT / haplen in float and double (avx-pairhmm-template.h:86,151).
//   tasks          one warp-task = up to 32/W reads x a run of consecutive haplotypes (see Task).
//   raw            float [pairs], read-major per region: the raw scaled likelihoods the reference's accelerator
//                  returns (task/xlnx/PairHMMTask.cpp:69-79).
//   fallback list  device-built tasks for pairs with raw < 1e-28f (PairHMMWorker.cpp:176), + their double results.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "pmm_types.h"

namespace pmm {

constexpr uint8_t kSep = 0xFF;          // separator element of the hap stream
constexpr int kStreamFrontPad = 64;     // bytes before stream[0] that lanes may read (and ignore) while filling
constexpr int kStreamTailPad = 128;



struct DeviceTables {
    const float*  ph2pr_f;
    const float*  m2m_f;
    const double* ph2pr_d;
    const double* m2m_d;
};

struct ForwardArgs {
    const uint8_t*  read_blob;
    const ReadDesc* reads;
    const float*    params;        // float pass: row parameters written by read_params_kernel (GroupDesc layout)
    const uint8_t*  stream;        // points at stream[0]; kStreamFrontPad readable bytes precede it
    const uint32_t* spos;          // [num_hap + 1]; spos[num_hap] = position of the final SEP
    const void*     inity;         // float* or double* [num_hap]
    const uint32_t* hap_list;      // double re-run: the tasks' haplotypes (Task::hap_first indexes this list)
    const Task*     tasks;
    const uint32_t* ntasks_dev;    // if non-null the task count is read from device memory (fallback list)
    uint32_t        ntasks;
    uint32_t*       counter;       // work-queue cursor, zeroed before launch
    void*           out;           // float* or double*
    void*           scratch;       // STRIPED only: per-warp carry rows, 3 * scratch_stride elements per warp
    uint32_t        scratch_stride;
    double          tiny_threshold;   // double kernel: results below it are re-run with flush-to-zero emulated ...
    uint32_t*       tiny_count;       // ... and counted here
    DeviceTables    tab;
};

// What the float pass reports about results below 1e-28f (PairHMMWorker.cpp:176): their number (the pairs themselves
// are found again by fallback_scan_kernel) and, in fast mode, the pairs too close to the threshold to decide.
struct FallbackQueue {
    uint32_t* reserve;       // results below `lo` so far (== fallback count when the float pass is done)
    uint32_t  capacity;      // room in recheck_tasks
    // Thresholds of the float pass: result < lo -> fallback list; lo <= result < hi -> exact re-check list.  Exact
    // kernels run with lo == hi == 1e-28f (the reference's test, PairHMMWorker.cpp:176); fast kernels with a guard band.
    float     lo, hi;
    Task*     recheck_tasks;
    uint32_t* recheck_count;
};

// Input of the two fallback-building kernels: they turn the results below the threshold into tasks for the double
// kernel, the failing haplotypes of one read together, longest tasks first.  ctrl: [0] number of failing pairs (counted
// by the float pass), [3] tasks written, [4] slots handed out, [kCtrlHist ..) tasks per cost class,
// [kCtrlClassCursor ..) write cursor of each class.
constexpr int kCostClasses = 64;
constexpr int kCtrlHist = 64, kCtrlClassCursor = 128, kCtrlCursors = 256;   // kCtrlCursors + 32 k: work-queue cursor of launch k
struct FallbackBuild {
    const float*      raw;
    const RegionDesc* regions;
    const ReadDesc*   reads;
    uint32_t          num_region, num_rows;
    float             threshold;
    uint32_t*         ctrl;
    Task*             tasks;
    uint32_t*         out_index;           // [slot] position of the pair in the job's result
    uint32_t*         hap_list;            // [slot] its haplotype
    uint32_t*         row_slot;            // [2 row] first slot and number of failing pairs of the row (scan -> tasks)
    const uint32_t*   spos;                // haplotype stream positions (lengths, for the task cost)
    uint32_t          max_hap_len;
    uint32_t          capacity;            // slots available (= pairs of the job)
    uint32_t          single_stripe_rows;  // 32 * K of the double kernel: longer reads get single-pair tasks
    uint32_t          target_tasks;        // tasks wanted: haplotypes per task = failing pairs / target_tasks ...
    uint32_t          max_run;             // ... but at most this many
};
cudaError_t launch_build_fallback(const FallbackBuild& b, int sm_count, cudaStream_t s);   // two launches

// Launch helpers implemented in pmm_kernels.cu -------------------------------------------------------------

// One instantiated variant of the forward kernel: CTAs per SM it reaches (0 if unknown) and its launch on `ctas` CTAs.
struct ForwardKernel {
    int (*ctas_per_sm)();
    cudaError_t (*launch)(const ForwardArgs& a, const FallbackQueue& fq, int ctas, cudaStream_t s);
};
// Float pass.  (K rows per lane) x (W lanes per read); W in {8,16,32}; null for an uninstantiated (K, W).  `striped`
// selects the multi-stripe variant for reads longer than W*K - 1 bases.  Results below 1e-28f are appended to fq.
const ForwardKernel* forward_f32_variant(int K, int W, bool striped, bool fast);
// Exact float re-run of the single-pair tasks on the re-check list (fast mode), overwriting their results.
const ForwardKernel& recheck_f32_variant();
// Double re-run (fq unused) of the tasks fallback_tasks_kernel wrote, K from pick_f64_rows(); null for a K not in kF64Rows.
// Results below a.tiny_threshold are recomputed in the same kernel with x86 flush-to-zero emulated on every product.
const ForwardKernel* forward_f64_variant(int K, bool striped);
int pick_f64_rows(uint32_t max_read_len);

cudaError_t launch_build_stream(const uint8_t* hap_blob, const HapDesc* haps, const uint32_t* spos, uint32_t num_hap,
                                uint8_t* stream, float* inity_f, double* inity_d, float ic_f, double ic_d,
                                cudaStream_t s);

// Row parameters of the float pass, one CTA per read group (layout: GroupDesc in pmm_types.h).
cudaError_t launch_read_params(const uint8_t* read_blob, const ReadDesc* reads, const GroupDesc* groups, uint32_t ngroups,
                               const DeviceTables& tab, float* params, cudaStream_t s);

// FP32 issue-rate probe used for the roofline denominator (dependent-free FMUL/FADD streams).
cudaError_t launch_fp32_probe(float* sink, int iters, int ctas, cudaStream_t s);
// The same for the FP64 pipe (independent DMUL/DADD streams): denominator of the double re-run's roofline.
cudaError_t launch_fp64_probe(double* sink, int iters, int ctas, cudaStream_t s);

}  // namespace pmm
