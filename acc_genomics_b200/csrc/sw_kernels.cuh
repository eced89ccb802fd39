// sw_kernels.cuh -- device-side data model of the Smith-Waterman aligner (shared by sw_kernels.cu and sw_engine.cu).
//
// Layout in HBM for one chunk of pairs:
//   seq1 / seq2 blobs   bytes; pair p is seq1[s1 .. s1+l1) (reference, matrix rows) against seq2[s2 .. s2+l2) (alternate, columns)
//   backtrack           per pair ceil(l1 / (32 K)) blocks of 32 K rows (K = rows_per_lane), every row `bt_stride` 32-bit words,
//                       laid out [block][word][lane][row of the lane] so that the fill's stores cover whole sectors;
//                       8 cells per word, 4 bits per cell: bit 3 "the insertion
//                       into this cell opens a gap" (else it extends one), bit 2 the same for the deletion, bit 1 "the
//                       insertion beats the diagonal", bit 0 "the deletion beats both" -- the information of the reference's
//                       codes (/root/reference/htc-sw/intel_avx/smithwaterman_common.h:18-22) as raw comparison results.
//                       Words are indexed by wavefront step: row i, column j is nibble 7 - (t & 7) of word t >> 3 with
//                       t = j - 1 + lane(i), lane(i) = ((i - 1) / rows_per_lane) % 32 (see sw_kernels.cu)
//   cigars              per pair `cigar_cap` (length, state) elements, forward order; n_elem, alignment offset, score
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace sw {

constexpr int kWarpsPerCta = 4;
constexpr int kMaxLen = 4095;
constexpr int kMaxWeight = 1 << 16;      // |match|, |mismatch|, |open|, |extend| at most this (see cells() in sw_kernels.cu)

struct PairDesc {
    uint32_t s1, l1, s2, l2;
    uint64_t bt_off;                     // first word of the pair's backtrack matrix
    uint32_t bt_stride;                  // words per row = ceil((l2 + 31) / 8)
    uint32_t index;                      // position of the pair in the caller's arrays
    uint32_t rows_per_lane;              // K of the fill: a block of rows = 32 lanes x K rows (pick_rows_per_lane)
    uint32_t pad_;
};

struct Args {
    const uint8_t*  seq1;
    const uint8_t*  seq2;
    const PairDesc* pairs;
    uint32_t        npairs;
    uint32_t*       counter;             // work-queue cursor, zero at launch
    uint32_t*       bt;
    int             match, mismatch, open, extend, strategy;
    uint32_t        cigar_cap;
    int2*           cigars;              // (length, state): per pair of the chunk a scratch row of cigar_cap elements (backward order)
    int2*           compact;             // forward-order CIGARs of all pairs back to back, in completion order
    uint32_t        compact_cap;         // room in `compact`; appends beyond it are counted but not written
    uint32_t*       compact_count;       // elements in `compact` so far (zero at the first launch of a batch)
    uint32_t*       compact_first;       // per pair: where its CIGAR starts in `compact`
    int32_t*        n_elem;
    int32_t*        offset;
    int32_t*        score;
    uint32_t        max_l1, max_l2;      // of the chunk: sizes the per-warp shared memory
    int             k_neg1, k_one;       // -1 and 1: multipliers kept opaque to the compiler (see cells() in sw_kernels.cu)
};

size_t smem_bytes_per_warp(uint32_t max_l1, uint32_t max_l2);
uint32_t pick_rows_per_lane(uint32_t l1);
cudaError_t launch_align(const Args& a, int sm_count, cudaStream_t s, int* ctas_out);

}  // namespace sw
