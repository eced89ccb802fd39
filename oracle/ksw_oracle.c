/* ksw_oracle.c -- CPU restatement of BWA-MEM's seed extension, ksw_extend2 of bwa 0.7.17 (ksw.c, MIT licence).
 * TEST INFRASTRUCTURE ONLY: nothing in the product links or calls this file.
 *
 * There is no copy of bwa in this repository.  The recurrence below is restated from bwa's published source and is the
 * contract sw_extend_batch (include/smithwaterman_cuda.h) is held to; it has not been checked against a bwa binary.
 * It is a literal transcription: a banded, integer, affine-gap DP over one row array eh[0..qlen] of {H, E}, with E and
 * F computed from M alone (bwa forbids CIGARs such as 3I3D that way), the band shrunk to the non-zero cells after
 * every row, the run stopped by an all-zero row or by the Z-drop test.  The reference's FPGA counterpart is
 * bwa-sw/sdaccel/smithwaterman.cpp (sw_core).
 *
 * Besides bwa's outputs it reports the number of DP cells its inner loop visited.
 */
#include <stdint.h>
#include <stdlib.h>

typedef struct { int32_t h, e; } eh_t;

/* out[0..5] = score, qle, tle, gtle, gscore, max_off; *cells = inner-loop iterations.  Returns score. */
int ksw_oracle_extend(int qlen, const uint8_t* query, int tlen, const uint8_t* target, int m, const int8_t* mat,
                      int o_del, int e_del, int o_ins, int e_ins, int w, int end_bonus, int zdrop, int h0,
                      int32_t* out, uint64_t* cells)
{
    eh_t* eh;
    int8_t* qp;
    int i, j, k, oe_del = o_del + e_del, oe_ins = o_ins + e_ins, beg, end, max, max_i, max_j, max_ins, max_del, max_ie,
        gscore, max_off;
    uint64_t n_cells = 0;
    qp = (int8_t*)malloc((size_t)qlen * m);
    eh = (eh_t*)calloc((size_t)qlen + 1, 8);
    /* query profile */
    for (k = i = 0; k < m; ++k) {
        const int8_t* p = &mat[k * m];
        for (j = 0; j < qlen; ++j) qp[i++] = p[query[j]];
    }
    /* first row */
    eh[0].h = h0; eh[1].h = h0 > oe_ins ? h0 - oe_ins : 0;
    for (j = 2; j <= qlen && eh[j - 1].h > e_ins; ++j) eh[j].h = eh[j - 1].h - e_ins;
    /* band cap */
    k = m * m;
    for (i = 0, max = 0; i < k; ++i) max = max > mat[i] ? max : mat[i];
    max_ins = (int)((double)(qlen * max + end_bonus - o_ins) / e_ins + 1.);
    max_ins = max_ins > 1 ? max_ins : 1;
    w = w < max_ins ? w : max_ins;
    max_del = (int)((double)(qlen * max + end_bonus - o_del) / e_del + 1.);
    max_del = max_del > 1 ? max_del : 1;
    w = w < max_del ? w : max_del;
    /* DP */
    max = h0, max_i = max_j = -1; max_ie = -1, gscore = -1;
    max_off = 0;
    beg = 0, end = qlen;
    for (i = 0; i < tlen; ++i) {
        int t, f = 0, h1, mm = 0, mj = -1;
        const int8_t* q = &qp[target[i] * qlen];
        if (beg < i - w) beg = i - w;
        if (end > i + w + 1) end = i + w + 1;
        if (end > qlen) end = qlen;
        if (beg == 0) {
            h1 = h0 - (o_del + e_del * (i + 1));
            if (h1 < 0) h1 = 0;
        } else h1 = 0;
        for (j = beg; j < end; ++j) {
            eh_t* p = &eh[j];
            int h, M = p->h, e = p->e;   /* H(i-1,j-1), E(i,j) */
            p->h = h1;                   /* H(i,j-1) for the next row */
            M = M ? M + q[j] : 0;
            h = M > e ? M : e;
            h = h > f ? h : f;
            h1 = h;
            mj = mm > h ? mj : j;        /* ties: the last column wins */
            mm = mm > h ? mm : h;
            t = M - oe_del;
            t = t > 0 ? t : 0;
            e -= e_del;
            e = e > t ? e : t;
            p->e = e;                    /* E(i+1,j) */
            t = M - oe_ins;
            t = t > 0 ? t : 0;
            f -= e_ins;
            f = f > t ? f : t;           /* F(i,j+1) */
            ++n_cells;
        }
        eh[end].h = h1; eh[end].e = 0;
        if (j == qlen) {
            max_ie = gscore > h1 ? max_ie : i;
            gscore = gscore > h1 ? gscore : h1;
        }
        if (mm == 0) break;
        if (mm > max) {
            max = mm, max_i = i, max_j = mj;
            max_off = max_off > abs(mj - i) ? max_off : abs(mj - i);
        } else if (zdrop > 0) {
            if (i - max_i > mj - max_j) {
                if (max - mm - ((i - max_i) - (mj - max_j)) * e_del > zdrop) break;
            } else {
                if (max - mm - ((mj - max_j) - (i - max_i)) * e_ins > zdrop) break;
            }
        }
        for (j = beg; j < end && eh[j].h == 0 && eh[j].e == 0; ++j) ;
        beg = j;
        for (j = end; j >= beg && eh[j].h == 0 && eh[j].e == 0; --j) ;
        end = j + 2 < qlen ? j + 2 : qlen;
    }
    free(eh); free(qp);
    out[0] = max; out[1] = max_j + 1; out[2] = max_i + 1; out[3] = max_ie + 1; out[4] = gscore; out[5] = max_off;
    if (cells) *cells = n_cells;
    return max;
}

/* Jobs one after another on the calling thread: job k is query[jobs[7k] .. +jobs[7k+1]) against
 * target[jobs[7k+2] .. +jobs[7k+3]) with h0, w, end_bonus = jobs[7k+4 .. 7k+6] (the layout of sw_extend_job_t).
 * out[6k .. 6k+5] as ksw_oracle_extend; cells[k] its cell count. */
void ksw_oracle_extend_batch(int n, const uint8_t* query, const uint8_t* target, const int32_t* jobs, int m,
                             const int8_t* mat, int o_del, int e_del, int o_ins, int e_ins, int zdrop, int32_t* out,
                             uint64_t* cells)
{
    for (int k = 0; k < n; ++k) {
        const int32_t* jb = jobs + 7 * (size_t)k;
        ksw_oracle_extend(jb[1], query + (uint32_t)jb[0], jb[3], target + (uint32_t)jb[2], m, mat, o_del, e_del, o_ins,
                          e_ins, jb[5], jb[6], zdrop, jb[4], out + 6 * (size_t)k, cells + k);
    }
}
