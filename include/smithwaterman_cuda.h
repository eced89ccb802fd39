/*
 * smithwaterman_cuda.h -- C ABI of the B200 Smith-Waterman aligner with backtrack (same library, libpairhmm_b200.so).
 *
 * This is row (f)4 of SURVEY.md section 8: the stage next to PairHMM in GATK HaplotypeCaller, where every candidate
 * haplotype is aligned to the reference window and the alignment is returned as a CIGAR.  It replaces, for that path,
 * the reference's CPU and FPGA implementations under /root/reference/htc-sw:
 *   - runSWOnePairBT_fp_avx2(match, mismatch, open, extend, seq1, seq2, len1, len2, overhangStrategy, Cigar*)
 *     (intel_avx/avx2_impl.h:6, intel_avx/PairWiseSW.h:441-470) -- one pair, returns the alignment offset;
 *   - SWPairwiseAlignmentMultiBatch(ref, refLength, alts, batchSize, altLengths, cigarResults, alignmentOffsets,
 *     overhang_strategy, option) (host/FalconSW_AVX.cpp:304-313) -- one reference against a batch of alternates;
 *   - FalconSWFPGA_run(...) / _smithWatermanRun(...) (host/sw_host.cpp:13, host/smithWatermanHost.h:14) -- the FPGA dispatch.
 * Results (alignment offset, CIGAR elements in forward order) are identical to those functions: integer arithmetic,
 * same tie-breaks in the cell update, in the search for the end cell and in the traceback.
 *
 * seq1 is the reference (rows of the matrix), seq2 the alternate (columns).  Bases are compared as bytes.  Sequences of
 * length 0 are rejected (the reference reads uninitialised memory for them).  CIGAR states are those of
 * host/common.h:20-23: 0 = M, 1 = I, 2 = D, 4 = S.  No CPU fallback: without a B200 every call fails.
 */
#ifndef SMITHWATERMAN_CUDA_H
#define SMITHWATERMAN_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct sw_ctx sw_ctx;

enum { SW_OK = 0, SW_ERR_INVALID = 1, SW_ERR_CUDA = 2, SW_ERR_NO_DEVICE = 3 };

/* overhang strategies (host/common.h:11-14) */
enum { SW_OVERHANG_SOFTCLIP = 0, SW_OVERHANG_INDEL = 1, SW_OVERHANG_LEADING_INDEL = 2, SW_OVERHANG_IGNORE = 3 };

/* Same layout as struct CigarElement (host/common.h:47-50). */
typedef struct { int32_t length; int32_t state; } sw_cigar_elem_t;

typedef struct {
    uint64_t pairs, cells;            /* cells = sum over pairs of len1 * len2 (host/FalconSW_AVX.cpp:316)   */
    uint64_t bytes_backtrack;         /* device memory used for the 4-bit backtrack matrices                  */
    uint32_t kernel_launches, chunks; /* a batch whose backtrack matrices exceed the budget runs in chunks    */
    float    ms_kernel, ms_total;     /* CUDA-event time of the kernels / wall time of the call               */
} sw_stats_t;

int  sw_create(int device, sw_ctx** out);         /* device < 0: the current one */
void sw_destroy(sw_ctx* ctx);
const char* sw_last_error(const sw_ctx* ctx);     /* ctx may be NULL: last error of sw_create */

/* Align n_pairs pairs.  Pair p is seq1_bytes[seq1_start[p] .. +seq1_len[p]) against seq2_bytes[seq2_start[p] .. +seq2_len[p])
 * (several pairs may name the same reference bytes).  Outputs, all caller-owned host memory:
 *   cigars[p * cigar_cap .. ]  the CIGAR elements of pair p in forward order, at most cigar_cap of them; only the first
 *                              min(n_elem[p], cigar_cap) elements of a row are written, the rest is left as it was.
 *                              When n_elem[p] > cigar_cap the row holds the LAST cigar_cap elements of the CIGAR, in
 *                              forward order (the traceback runs from the end of the alignment): retry larger
 *   n_elem[p]                  how many elements the CIGAR has
 *   alignment_offset[p]        the value runSWOnePairBT returns / SWPairwiseAlignmentOneBatch stores
 *   score[p]                   (optional, may be NULL) the score H of the cell where the traceback starts.  For SOFTCLIP,
 *                              INDEL and LEADING_INDEL that is the score of the returned alignment: match / mismatch per
 *                              M base, open + (L - 1) * extend per I or D element of length L, 0 per S base (exact
 *                              unless the -10^8 clamp below acts, or open > extend lets two gaps touch and merge into
 *                              one element).  For IGNORE it is the score of the end cell the search found
 * Weights are the reference's W_MATCH, W_MISMATCH, W_OPEN, W_EXTEND (host/common.h:15-18: 200, -150, -260, -11 by default
 * in GATK), each within [-65536, 65536] (else SW_ERR_INVALID): then no score can overflow 32 bits.  Any sign is accepted.
 * Limits: each sequence at most 4095 bases.  Like the reference, the diagonal term of the recurrence is clamped at
 * -10^8 (MATRIX_MIN_CUTOFF); within the weight domain that clamp can act (e.g. mismatch <= -24415 at 4095 bases). */
int  sw_align_batch(sw_ctx* ctx, uint32_t n_pairs,
                    const uint8_t* seq1_bytes, const uint32_t* seq1_start, const uint32_t* seq1_len,
                    const uint8_t* seq2_bytes, const uint32_t* seq2_start, const uint32_t* seq2_len,
                    int w_match, int w_mismatch, int w_open, int w_extend, int overhang_strategy,
                    uint32_t cigar_cap, sw_cigar_elem_t* cigars, int32_t* n_elem, int32_t* alignment_offset, int32_t* score);

int  sw_get_stats(const sw_ctx* ctx, sw_stats_t* out);

#ifdef __cplusplus
}
#endif
#endif /* SMITHWATERMAN_CUDA_H */
