/* sw_oracle.c -- CPU restatement of the reference's Smith-Waterman with backtrack (haplotype-to-reference alignment
 * of GATK HaplotypeCaller).  TEST INFRASTRUCTURE ONLY: nothing in the product links or calls this file.
 *
 * Follows /root/reference/htc-sw/intel_avx/PairWiseSW.h: the recurrence and backtrack codes of MAIN_CODE (:4-40),
 * boundary values (:218-228), the search for the end cell with its tie-breaks (:233-262), and getCIGAR (:275-437).
 * Plain scalar C over full (len1+1) x (len2+1) matrices; the reference sweeps anti-diagonals with AVX2, which only
 * changes the order in which independent cells are visited -- except for the end-cell search, whose order of visits
 * matters and is reproduced here (anti-diagonal by anti-diagonal, last row before last column).
 *
 * seq1 = reference (rows, index i), seq2 = alternate (columns, index j).  Cigar states: 0 M, 1 I, 2 D, 4 S
 * (host/common.h:20-23).  Returns the alignment offset; the cigar comes out in forward order as (length, state) pairs,
 * and *score_out is H of the cell the traceback starts from (for IGNORE: the end cell of the search).
 */
#include <limits.h>
#include <stdint.h>
#include <stdlib.h>

#define BT_MATCH 0
#define BT_INSERT 1
#define BT_DELETE 2
#define BT_INSERT_EXT 4
#define BT_DELETE_EXT 8
#define OP_SOFTCLIP 9              /* internal code of getCIGAR (smithwaterman_common.h:23) */
#define STRAT_SOFTCLIP 0
#define STRAT_INDEL 1
#define STRAT_LEADING_INDEL 2
#define STRAT_IGNORE 3
#define MATRIX_MIN_CUTOFF (-100000000)
#define LOW_INIT_VALUE (INT32_MIN / 2)

static int iabs(int x) { return x < 0 ? -x : x; }

int sw_oracle_align(int match, int mismatch, int open, int extend, const uint8_t* seq1, int nrow, const uint8_t* seq2,
                    int ncol, int strategy, int* cigar_len, int* cigar_state, int cigar_cap, int* n_elem, int* score_out)
{
    const int W = ncol + 1;
    int32_t* H = (int32_t*)malloc(sizeof(int32_t) * (size_t)(nrow + 1) * W);
    int32_t* E = (int32_t*)malloc(sizeof(int32_t) * (size_t)(nrow + 1) * W);   /* gap along the row: consumes seq2 (insertion) */
    int32_t* F = (int32_t*)malloc(sizeof(int32_t) * (size_t)(nrow + 1) * W);   /* gap along the column: consumes seq1 (deletion) */
    uint8_t* B = (uint8_t*)calloc((size_t)(nrow + 1) * W, 1);
    int i, j;
    const int indel = strategy == STRAT_INDEL || strategy == STRAT_LEADING_INDEL;
    /* boundaries (PairWiseSW.h:218-228; H[0][0] = 0 at :87) */
    for (i = 0; i <= nrow; ++i) { H[i * W] = (i && indel) ? open + (i - 1) * extend : 0; E[i * W] = LOW_INIT_VALUE; F[i * W] = LOW_INIT_VALUE; }
    for (j = 0; j <= ncol; ++j) { H[j] = (j && indel) ? open + (j - 1) * extend : 0; E[j] = LOW_INIT_VALUE; F[j] = LOW_INIT_VALUE; }
    /* cell update (MAIN_CODE, :4-40) */
    for (i = 1; i <= nrow; ++i)
        for (j = 1; j <= ncol; ++j) {
            const int32_t ext_h = E[i * W + j - 1] + extend, open_h = H[i * W + j - 1] + open;
            const int32_t e11 = open_h > ext_h ? open_h : ext_h;
            int bt_ext = open_h > ext_h ? 0 : BT_INSERT_EXT;
            const int32_t ext_v = F[(i - 1) * W + j] + extend, open_v = H[(i - 1) * W + j] + open;
            const int32_t f11 = ext_v > open_v ? ext_v : open_v;
            if (!(open_v > ext_v)) bt_ext |= BT_DELETE_EXT;
            const int32_t m11 = H[(i - 1) * W + j - 1] + (seq1[i - 1] == seq2[j - 1] ? match : mismatch);
            int32_t h11 = m11 > MATRIX_MIN_CUTOFF ? m11 : MATRIX_MIN_CUTOFF;
            int bt = BT_MATCH;
            if (e11 > h11) { bt = BT_INSERT; h11 = e11; }
            if (f11 > h11) { bt = BT_DELETE; h11 = f11; }
            E[i * W + j] = e11; F[i * W + j] = f11; H[i * W + j] = h11; B[i * W + j] = (uint8_t)(bt | bt_ext);
        }
    /* end cell (:233-262): anti-diagonals in ascending order; on each, the last-row cell first, then the last-column cell */
    int32_t max_score = INT32_MIN; int max_i = 0, max_j = 0, update_max_j = 0;
    for (int ad = 1; ad <= nrow + ncol; ++ad) {
        if (ad >= nrow + 1) {                                  /* touches the last row: cell (nrow, ad - nrow) */
            const int jj = ad - nrow;
            if (jj >= 1 && jj <= ncol && (strategy == STRAT_SOFTCLIP || strategy == STRAT_IGNORE)) {
                const int32_t s = H[nrow * W + jj];
                if (max_score < s || (max_score == s && iabs(nrow - jj) < iabs(max_i - max_j))) { max_score = s; max_i = nrow; max_j = jj; update_max_j = 1; }
            }
        }
        if (ad >= ncol + 1) {                                  /* touches the last column: cell (ad - ncol, ncol) */
            const int ii = ad - ncol;
            if (ii >= 1 && ii <= nrow) {
                const int32_t s = H[ii * W + ncol];
                if (max_score < s || (max_score == s && (max_j == ncol || iabs(ii - ncol) <= iabs(max_i - max_j)))) { max_score = s; max_i = ii; max_j = ncol; update_max_j = 1; }
            }
        }
    }
    /* the score of the cell the traceback starts from (INDEL: the corner, whatever the search found) */
    if (score_out) *score_out = strategy == STRAT_INDEL ? H[nrow * W + ncol] : max_score;

    /* traceback (getCIGAR, :275-437) */
    int* ops = (int*)malloc(sizeof(int) * 2 * (size_t)(nrow + ncol + 4));
    int n = 0, segment_length = 0, offset = 0;
    if (strategy == STRAT_INDEL) { i = nrow; j = ncol; }
    else if (strategy == STRAT_LEADING_INDEL) { i = max_i; j = ncol; }
    else { i = max_i; j = max_j; }
    if (j < ncol && strategy == STRAT_SOFTCLIP) { ops[2 * n] = OP_SOFTCLIP; ops[2 * n + 1] = ncol - j; ++n; }
    if (strategy == STRAT_IGNORE && update_max_j && j != ncol) { i = nrow; segment_length = ncol - max_j; }
    int state = 0;
    while (i > 0 && j > 0) {
        const int btr = B[i * W + j];
        if (state == BT_INSERT_EXT) { --j; ops[2 * n - 1]++; state = btr & BT_INSERT_EXT; }
        else if (state == BT_DELETE_EXT) { --i; ops[2 * n - 1]++; state = btr & BT_DELETE_EXT; }
        else switch (btr & 3) {
            case BT_MATCH:
                --i; --j; ops[2 * n] = BT_MATCH;
                ops[2 * n + 1] = (n == 0 && strategy == STRAT_IGNORE) ? segment_length + 1 : 1;
                state = 0; ++n; break;
            case BT_INSERT: --j; ops[2 * n] = BT_INSERT; ops[2 * n + 1] = 1; state = btr & BT_INSERT_EXT; ++n; break;
            case BT_DELETE: --i; ops[2 * n] = BT_DELETE; ops[2 * n + 1] = 1; state = btr & BT_DELETE_EXT; ++n; break;
            default: state = 0; break;                          /* code 3 does not occur */
        }
    }
    if (strategy == STRAT_SOFTCLIP) {
        if (j > 0) { ops[2 * n] = OP_SOFTCLIP; ops[2 * n + 1] = j; ++n; }
        offset = i;
    } else if (strategy == STRAT_IGNORE) {
        if (j > 0) { ops[2 * n] = n ? ops[2 * (n - 1)] : 0; ops[2 * n + 1] = j; ++n; }
        offset = i - j;
    } else {
        if (i > 0) { ops[2 * n] = BT_DELETE; ops[2 * n + 1] = i; ++n; }
        else if (j > 0) { ops[2 * n] = BT_INSERT; ops[2 * n + 1] = j; ++n; }
        offset = 0;
    }
    /* merge equal neighbours, then reverse into forward order (:404-436) */
    int m = 0;
    for (int k = 1; k < n; ++k) {
        if (ops[2 * k] == ops[2 * m]) ops[2 * m + 1] += ops[2 * k + 1];
        else { ++m; ops[2 * m] = ops[2 * k]; ops[2 * m + 1] = ops[2 * k + 1]; }
    }
    int count = n ? m + 1 : 0, w = 0;
    for (int k = count - 1; k >= 0 && w < cigar_cap; --k, ++w) {
        cigar_len[w] = ops[2 * k + 1];
        cigar_state[w] = ops[2 * k] == OP_SOFTCLIP ? 4 : ops[2 * k];
    }
    *n_elem = count;
    free(ops); free(H); free(E); free(F); free(B);
    return offset;
}
