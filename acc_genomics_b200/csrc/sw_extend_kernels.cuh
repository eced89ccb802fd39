// sw_extend_kernels.cuh -- device-side data model of the BWA-MEM seed extension (sw_extend_kernels.cu, sw_engine.cu).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace swx {

constexpr int kWarpsPerCta = 4;
constexpr int kMaxQuery = 4095, kMaxTarget = 65535, kMaxAlphabet = 16;
constexpr int kMaxH0 = 1 << 24, kMaxGap = 4096, kMaxBand = 65535, kMaxEndBonus = 65536;

struct JobDesc {
    uint32_t q_start, q_len, t_start, t_len;
    int32_t  h0;
    int32_t  w;                          // the band after bwa's cap (computed on the host, in double like bwa)
    uint32_t index;                      // position of the job in the caller's arrays
    uint32_t pad_;
};

struct Args {
    const uint8_t* query;
    const uint8_t* target;
    const JobDesc* jobs;                 // largest first
    uint32_t       njobs;
    uint32_t*      counter;              // work-queue cursor, zero at launch
    int32_t*       out;                  // 6 int32 per job, at the job's index
    unsigned long long* cells;           // DP cells visited, summed over the batch (zero at launch)
    uint32_t       max_qlen;             // sizes the per-warp shared memory
    int            m, o_del, e_del, o_ins, e_ins, zdrop;
    int8_t         mat[kMaxAlphabet * kMaxAlphabet];
};

cudaError_t launch_extend(const Args& a, int sm_count, cudaStream_t s);

}  // namespace swx
