// sw_kernels.cu -- sm_100a Smith-Waterman with backtrack: matrix fill, end-cell search and traceback in one kernel.
//
// The arithmetic and every tie-break are those of the reference's AVX2 kernel
// (/root/reference/htc-sw/intel_avx/PairWiseSW.h: MAIN_CODE :4-40, boundaries :218-228, end cell :233-262, getCIGAR
// :275-437), which Falcon's own SWPairwiseAlignmentOneBatch (host/FalconSW_AVX.cpp:315-411, :2303-2415) agrees with.
//
// Mapping to the machine:
//   * One warp aligns one pair.  The matrix is processed in blocks of 32 x kRowsPerLane rows: lane l owns kRowsPerLane
//     consecutive rows and sweeps the columns, skewed by one column per lane, so the lane above has always just
//     finished the column a lane is about to do (the same wavefront as the PairHMM kernel).  H and F of the row above
//     a lane's first row arrive by two __shfl_up_sync per step; H of a lane's own rows, and E, stay in registers.
//   * The last row of a block is carried to the next block through a per-warp row in shared memory (written by lane 31,
//     read 31 steps earlier by lane 0 -- one buffer is enough).  The alternate sequence, the last row / last column of H
//     (for the end-cell search) and the traceback tile live in shared memory too.
//   * Backtrack codes are packed 8 cells per 32-bit word per row; a lane completes one word per row every 8 steps.  The
//     words of a block of rows are laid out [word][lane][row of the lane], so the K words a lane stores at such a step
//     are contiguous and the warp's stores cover whole sectors; the traceback fetches a 32-row x 64-column tile as nine
//     words per row, the rows of one lane next to each other.
//   * The traceback is a pointer chase, but most of it is runs of diagonal moves: all lanes fetch a tile of codes, lane r
//     looks r cells down the diagonal and a ballot finds how far the run goes (one iteration per run or gap cell).
#include "sw_kernels.cuh"

#include <climits>

namespace sw {
namespace {

constexpr int kLowInit = INT32_MIN / 2;          // LOW_INIT_VALUE (smithwaterman_common.h:52)
constexpr int kMinCutoff = -100000000;           // MATRIX_MIN_CUTOFF (:51)
constexpr int kInsert = 1, kDelete = 2, kInsertExt = 4, kDeleteExt = 8;
constexpr int kStateClip = 4;                    // STATE_CLIP (host/common.h:23)
constexpr int kSoftClip = 0, kIndel = 1, kLeadingIndel = 2, kIgnore = 3;

// Integer multiply-add / high multiply as explicit PTX so that they stay IMAD / IMAD.HI (FMA pipe).
__device__ __forceinline__ int imad(int a, int b, int c)
{
    int d;
    asm("mad.lo.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

struct WarpSmem {
    int* carryH; int* carryF; int* lastrow; int* lastcol; uint32_t* tile; uint8_t* alt;
};

__host__ __device__ inline size_t align4(size_t x) { return (x + 3) & ~(size_t)3; }

__host__ __device__ inline size_t per_warp_bytes(uint32_t max_l1, uint32_t max_l2)
{
    const size_t c1 = align4(max_l2 + 1), r1 = align4(max_l1 + 1);
    const size_t b = sizeof(int) * (3 * c1 + r1) + sizeof(uint32_t) * 32 * 8 + align4(max_l2 + 4);
    return (b + 15) & ~(size_t)15;
}

__device__ __forceinline__ WarpSmem carve(char* base, uint32_t max_l1, uint32_t max_l2)
{
    WarpSmem w;
    const size_t c1 = align4(max_l2 + 1), r1 = align4(max_l1 + 1);
    w.carryH = reinterpret_cast<int*>(base);
    w.carryF = w.carryH + c1;
    w.lastrow = w.carryF + c1;
    w.lastcol = w.lastrow + c1;
    w.tile = reinterpret_cast<uint32_t*>(w.lastcol + r1);
    w.alt = reinterpret_cast<uint8_t*>(w.tile + 32 * 8);
    return w;
}

// Rows per lane available to the fill (a block of rows = 32 lanes x K rows).  The host picks K per pair so that the
// pair's rows fill its blocks (pick_rows_per_lane): a 375-row matrix takes one block of K = 12 (384 rows) instead of
// two of K = 8 (512 rows, and two fill/drain phases).
#define SW_ROWS_PER_LANE(X) X(4) X(6) X(8) X(10) X(12) X(14)
constexpr uint32_t kMaxRowsPerLane = 14;          // measured: 16 rows per lane are slower (501 vs 670 GCUPS), as are caps of 8..12

struct FillCtx {
    WarpSmem sm;
    const uint8_t* s1;
    uint32_t* B;
    uint32_t stride;
    int nrow, ncol, lane;
    int match, mismatch, open, extend;
    bool indel;
    int neg1;
};

// CUTOFF: apply max(MATRIX_MIN_CUTOFF, .) to the diagonal term like the reference (PairWiseSW.h:31).  The host drops it
// when the weights and lengths of the chunk cannot produce a score anywhere near -10^8 (see launch_align).
template <int K, bool CUTOFF>
__device__ __forceinline__ void fill_matrix(const FillCtx& c)
{
    const WarpSmem sm = c.sm;
    const int nrow = c.nrow, ncol = c.ncol, lane = c.lane;
    const int match = c.match, mismatch = c.mismatch, open = c.open, extend = c.extend;
    const bool indel = c.indel;
    const int neg1 = c.neg1;                       // -1, kept opaque to the compiler (see cells())
    {
        const int nblk = (nrow + 32 * K - 1) / (32 * K);
        #pragma unroll 1
        for (int blk = 0; blk < nblk; ++blk) {
            const int ifirst = blk * 32 * K + lane * K + 1;           // 1-based row of this lane's first row
            int Hrow[K], E[K];
            uint32_t acc[K];                                           // the last 8 steps' codes of each row, newest lowest
            int c1[K];
            #pragma unroll
            for (int k = 0; k < K; ++k) {
                const int i = ifirst + k;
                c1[k] = i <= nrow ? (int)c.s1[i - 1] : -1;
                Hrow[k] = indel ? open + (i - 1) * extend : 0;       // H[i][0]
                E[k] = kLowInit;
                acc[k] = 0;
            }
            // backtrack words of this block: [word][lane][row of the lane] -- the K words a lane completes at one step are
            // contiguous and the warp's 32 K words are one contiguous run, so every store fills whole 32-byte sectors
            // (row-major rows of words put each 4-byte store into a sector of its own: 2.5 x the bytes in DRAM writes)
            uint32_t* const bblk = c.B + ((size_t)blk * c.stride * 32 + lane) * K;
            int prev_up = (ifirst - 1 == 0) ? 0 : (indel ? open + (ifirst - 2) * extend : 0);   // H[ifirst-1][0]
            int lastF = kLowInit;
            // the lane and row that hold the matrix's last row (for the end-cell search); -1 if not in this block
            const int own_k = (nrow >= ifirst && nrow < ifirst + K) ? nrow - ifirst : -1;
            const bool blk_has_owner = __any_sync(0xffffffffu, own_k >= 0);
            const bool own_b0 = (own_k & 1) != 0, own_b1 = (own_k & 2) != 0, own_b2 = (own_k & 4) != 0, own_b3 = (own_k & 8) != 0;

            // Column j of this lane's K rows.  MAIN_CODE (PairWiseSW.h:4-40): same comparisons, same order.
            // Pipe balance: adds, min/max, compares, selects and shifts issue on the ALU pipe (half rate), multiply-adds
            // with at most two register operands on the FMA pipe.  Each of the four tie-breaks of a cell is the sign of a
            // difference (a multiply-add by a -1 ptxas cannot see through), and one funnel shift both extracts that sign
            // and appends it to the row's code word: acc = (acc << 1) | (diff >> 31).  Eight steps fill a word, older
            // codes fall off the top, nothing is ever reset or positioned.  Differences cannot overflow because the host
            // accepts only |weight| <= 2^16 and lengths <= 4095: every H, E and F is the score of a path of at most
            // 4095 + 4095 moves of one weight each (or the clamp, -10^8, in between), so |H|, |E|, |F| <= 8190 * 2^16
            // < 2^29; the one other operand is E or F of the boundary plus extend, kLowInit + extend, within
            // 2^30 + 2^16 of zero.  Every difference is then below 2^30 + 2^29 + 2^16 < 2^31 in magnitude.
            // History: compare + select + multiply-add packing with a per-step flush test, 40 instructions per cell,
            // 433 GCUPS; this form 24.
            auto cells = [&](const int j, const int c2, int upH, int upF) {
                int diag = prev_up;
                prev_up = upH;
                int hup = upH, fup = upF;
                #pragma unroll
                for (int k = 0; k < K; ++k) {
                    const int hleft = Hrow[k];
                    const int ext_h = E[k] + extend, open_h = hleft + open;
                    const int e11 = max(ext_h, open_h);
                    const int d_ins_open = imad(open_h, neg1, ext_h);           // < 0: open_h > ext_h; ties extend
                    const int ext_v = fup + extend, open_v = hup + open;
                    const int f11 = max(ext_v, open_v);
                    const int d_del_open = imad(open_v, neg1, ext_v);
                    const int m11 = diag + (c1[k] == c2 ? match : mismatch);
                    const int h0 = CUTOFF ? max(kMinCutoff, m11) : m11;
                    const int d_take_ins = imad(e11, neg1, h0);                 // < 0: e11 > h0
                    const int h1 = max(h0, e11);
                    const int d_take_del = imad(f11, neg1, h1);                 // < 0: f11 > h1
                    const int h11 = max(h1, f11);
                    uint32_t w = acc[k];
                    w = __funnelshift_l((uint32_t)d_ins_open, w, 1);
                    w = __funnelshift_l((uint32_t)d_del_open, w, 1);
                    w = __funnelshift_l((uint32_t)d_take_ins, w, 1);
                    w = __funnelshift_l((uint32_t)d_take_del, w, 1);
                    acc[k] = w;
                    diag = hleft;
                    Hrow[k] = h11; E[k] = e11; hup = h11; fup = f11;
                }
                lastF = fup;
                if (blk_has_owner) {                                    // warp-uniform: no reconvergence point in the loop
                    // Hrow[own_k] by a select tree on the bits of own_k (loop-invariant predicates, no compares)
                    int v[K];
                    #pragma unroll
                    for (int k = 0; k < K; ++k) v[k] = Hrow[k];
                    #pragma unroll
                    for (int bit = 0, n = K; n > 1; ++bit, n = (n + 1) / 2) {
                        const bool b = bit == 0 ? own_b0 : bit == 1 ? own_b1 : bit == 2 ? own_b2 : own_b3;
                        #pragma unroll
                        for (int m = 0; 2 * m < n; ++m) v[m] = (2 * m + 1 < n && b) ? v[2 * m + 1] : v[2 * m];
                    }
                    if (own_k >= 0) sm.lastrow[j] = v[0];
                }
                if (lane == 31) { sm.carryH[j] = Hrow[K - 1]; sm.carryF[j] = lastF; }
            };
            auto store_words = [&](const int word, const int shift) {
                static_assert(K % 2 == 0, "rows per lane are stored as 8-byte pairs");
                uint2* dst = reinterpret_cast<uint2*>(bblk + (size_t)word * 32 * K);     // rows past nrow: padding, allocated
                #pragma unroll
                for (int k = 0; k < K; k += 2) dst[k >> 1] = make_uint2(acc[k] << shift, acc[k + 1] << shift);
            };

            // Backtrack words are indexed by step, not by column: the code of row i, column j sits in word t >> 3 of the
            // row, nibble 7 - (t & 7), with t = j - 1 + (lane of row i).  All lanes then complete a word at the same
            // step, and the steady loop needs no test at all.
            const int steps = ncol + 31;
            int t = 0;
            // steps where some lanes have no column (fill, drain) or that do not line up with a word
            auto ragged = [&](const int tend) {
                #pragma unroll 1
                for (; t < tend; ++t) {
                    int upH = __shfl_up_sync(0xffffffffu, Hrow[K - 1], 1);
                    int upF = __shfl_up_sync(0xffffffffu, lastF, 1);
                    const int j = t - lane + 1;
                    if (j >= 1 && j <= ncol) {
                        if (lane == 0) { upH = sm.carryH[j]; upF = sm.carryF[j]; }
                        cells(j, (int)sm.alt[j - 1], upH, upF);
                        const int u = t & 7;
                        if (u == 7 || j == ncol) store_words(t >> 3, 4 * (7 - u));   // a row's last word: left-aligned
                    }
                }
            };
            if (ncol >= 40) {
                ragged(32);
                // The step body is kept once in the instruction stream (the funnel-shift packing needs no position, so
                // nothing forces an unroll): unrolled eight times it is 23 KB, streams through the instruction caches
                // and "no instruction" becomes the top stall (ncu: 1.0 per issued instruction).  Branch-free: every lane
                // reads the carry row at its own column and lane 0 keeps the value; the alternate base of the next
                // step is fetched one step ahead.
                const bool lane0 = lane == 0;
                int c2 = (int)sm.alt[t - lane];                        // column t - lane + 1
                #pragma unroll 1
                for (; t + 8 <= ncol; t += 8) {
                    #pragma unroll 1
                    for (int u = 0; u < 8; ++u) {
                        const int j = t + u - lane + 1;
                        const int sH = __shfl_up_sync(0xffffffffu, Hrow[K - 1], 1);
                        const int sF = __shfl_up_sync(0xffffffffu, lastF, 1);
                        const int cH = sm.carryH[j], cF = sm.carryF[j];
                        const int c2n = (int)sm.alt[j];                // next step's base (one slack byte past the end)
                        cells(j, c2, lane0 ? cH : sH, lane0 ? cF : sF);
                        c2 = c2n;
                    }
                    store_words(t >> 3, 0);
                }
            }
            ragged(steps);
            // H[i][ncol] of the lane's rows: still in registers, nothing touched them after the last column
            #pragma unroll
            for (int k = 0; k < K; ++k) if (ifirst + k <= nrow) sm.lastcol[ifirst + k] = Hrow[k];
            __syncwarp();
        }
    }
}

// Occupancy: three CTAs (12 warps) per SM with up to 168 registers beat four with 128 -- 670 against 510 GCUPS on 16 640
// pairs, 243 against 211 on one 260-pair batch (ptxas schedules the dependent chains better with the extra registers, and
// a fourth fill warp per SMSP only adds contention for the half-rate ALU pipe); two CTAs with 200 registers: 662.
template <bool CUTOFF>
__global__ void __launch_bounds__(kWarpsPerCta * 32, 3) sw_align_kernel(const Args a)
{
    extern __shared__ int4 smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const size_t per_warp = per_warp_bytes(a.max_l1, a.max_l2);
    const WarpSmem sm = carve(reinterpret_cast<char*>(smem_raw) + warp * per_warp, a.max_l1, a.max_l2);
    const int open = a.open, extend = a.extend, strategy = a.strategy;
    const bool indel = strategy == kIndel || strategy == kLeadingIndel;

    for (;;) {
        uint32_t p = 0;
        if (lane == 0) p = atomicAdd(a.counter, 1u);
        p = __shfl_sync(0xffffffffu, p, 0);
        if (p >= a.npairs) break;
        const PairDesc pd = a.pairs[p];
        const int nrow = (int)pd.l1, ncol = (int)pd.l2;
        const uint8_t* s2 = a.seq2 + pd.s2;
        uint32_t* B = a.bt + pd.bt_off;
        const uint32_t stride = pd.bt_stride;
        const int K = (int)pd.rows_per_lane;
        const uint32_t kdiv = ((1u << 20) + K - 1) / K;                 // (x * kdiv) >> 20 == x / K for x < 4096
        auto lane_of_row = [&](int row) { return (int)((((uint32_t)(row - 1) * kdiv) >> 20) & 31u); };
        // word w of a row in the [block][word][lane][row of the lane] layout of the backtrack matrix
        auto row_base = [&](int row) {
            const uint32_t q = ((uint32_t)(row - 1) * kdiv) >> 20;          // (row - 1) / K
            return B + ((size_t)(q >> 5) * stride * 32 + (q & 31u)) * K + ((uint32_t)(row - 1) - q * K);
        };

        __syncwarp();
        for (int x = lane; x < ncol; x += 32) sm.alt[x] = s2[x];
        // row 0: H[0][j] (PairWiseSW.h:218-228, H[0][0] = 0 at :87), F[0][j] = low
        for (int j = lane; j <= ncol; j += 32) {
            sm.carryH[j] = (j && indel) ? open + (j - 1) * extend : 0;
            sm.carryF[j] = kLowInit;
        }
        __syncwarp();

        // ---- matrix fill -----------------------------------------------------------------------------------------
        {
            const FillCtx fc{sm, a.seq1 + pd.s1, B, stride, nrow, ncol, lane, a.match, a.mismatch, open, extend, indel, a.k_neg1};
            switch (K) {
#define X(k) case k: fill_matrix<k, CUTOFF>(fc); break;
                SW_ROWS_PER_LANE(X)
#undef X
                default: break;                                         // the host only hands out the values above
            }
        }

        // ---- end cell (PairWiseSW.h:233-262): anti-diagonals ascending, last-row cell before last-column cell ----------
        // The reference scans the candidates one by one and keeps the first cell of the best score unless a later one of
        // the same score wins a tie-break against the cell held at that moment.  Cells below the final maximum can never
        // influence the outcome (the first cell that reaches it replaces whatever is held), so: the maximum by a warp
        // reduction, then only the cells that attain it, in the reference's order, 32 anti-diagonals per ballot.
        int ti = 0, tj = 0, seg = 0, best = INT32_MIN;
        int max_i = 0, max_j = 0;
        const bool updated = true;                 // some candidate is always taken: the last column has nrow >= 1 cells
        {
            const bool use_row = strategy == kSoftClip || strategy == kIgnore;
            for (int x = lane + 1; x <= nrow; x += 32) best = max(best, sm.lastcol[x]);
            if (use_row) for (int x = lane + 1; x <= ncol; x += 32) best = max(best, sm.lastrow[x]);
            #pragma unroll
            for (int d = 16; d; d >>= 1) best = max(best, __shfl_xor_sync(0xffffffffu, best, d));
            bool have = false;                      // a cell of the maximal score is held (same on every lane)
            for (int base = 1; base <= nrow + ncol; base += 32) {
                const int ad = base + lane, jj = ad - nrow, ii = ad - ncol;
                const bool rt = use_row && jj >= 1 && jj <= ncol && sm.lastrow[jj] == best;
                const bool ct = ii >= 1 && ii <= nrow && sm.lastcol[ii] == best;
                const unsigned rb = __ballot_sync(0xffffffffu, rt), cb = __ballot_sync(0xffffffffu, ct);
                for (unsigned any = rb | cb; any; any &= any - 1) {
                    const int l = __ffs((int)any) - 1, a2 = base + l;
                    if ((rb >> l) & 1u) {                                  // last-row cell (nrow, a2 - nrow) comes first
                        const int j2 = a2 - nrow;
                        if (!have || abs(nrow - j2) < abs(max_i - max_j)) { max_i = nrow; max_j = j2; have = true; }
                    }
                    if ((cb >> l) & 1u) {                                  // then the last-column cell (a2 - ncol, ncol)
                        const int i2 = a2 - ncol;
                        if (!have || max_j == ncol || abs(i2 - ncol) <= abs(max_i - max_j)) { max_i = i2; max_j = ncol; have = true; }
                    }
                }
            }
        }
        // start of the traceback (getCIGAR, :285-314); the walk's state is kept identical on all lanes
        if (strategy == kIndel) { ti = nrow; tj = ncol; }
        else if (strategy == kLeadingIndel) { ti = max_i; tj = ncol; }
        else { ti = max_i; tj = max_j; }
        if (strategy == kIgnore && updated && tj != ncol) { ti = nrow; seg = ncol - max_j; }

        // ---- traceback ------------------------------------------------------------------------------------------------------
        // A walk is a pointer chase (each move depends on the cell before), but most of it is runs of diagonal moves.  All
        // lanes fetch a 32-row x 64-column tile of codes, realigned from step-indexed words to column-indexed ones; then
        // lane r looks at the r-th cell down the diagonal from the current one and a ballot finds how far the diagonal run
        // goes -- one iteration per run or per gap cell instead of one per move (a 400-move walk: ~25 iterations).
        int2* out = a.cigars + (size_t)p * a.cigar_cap;              // scratch row of this pair within its chunk
        int n = 0;                         // elements written (run-length encoded, still in backward order)
        int cur_state = -1, cur_len = 0;   // the open run
        int raw_ops = 0;                   // getCIGAR's cigarId: number of un-merged operations so far
        int state = 0;
        auto emit = [&](int st, int len) {
            if (st == cur_state) { cur_len += len; return; }
            if (cur_state >= 0) { if (lane == 0 && (uint32_t)n < a.cigar_cap) out[n] = make_int2(cur_len, cur_state); ++n; }
            cur_state = st; cur_len = len;
        };
        if (tj < ncol && strategy == kSoftClip) { emit(kStateClip, ncol - tj); ++raw_ops; }
        while (ti > 0 && tj > 0) {
            const int ai = ti, aj = tj;
            const int cw0 = max(0, ((aj - 1) >> 3) - 7);               // first column-indexed word of the tile
            {
                // row ai - lane: nine step-indexed words starting at cw0 + (lane of the row) / 8, shifted left by
                // (lane of the row) % 8 codes, give the eight column-indexed words cw0 .. cw0 + 7
                const int row = ai - lane;
                const int lr = row >= 1 ? lane_of_row(row) : 0;
                const uint32_t* src = row_base(max(row, 1));
                const int w0 = cw0 + (lr >> 3), sh = 4 * (lr & 7);
                uint32_t raw[9];
                #pragma unroll
                for (int w = 0; w < 9; ++w) raw[w] = (row >= 1 && (uint32_t)(w0 + w) < stride) ? __ldcg(src + (size_t)(w0 + w) * 32 * K) : 0u;
                #pragma unroll
                for (int w = 0; w < 8; ++w) sm.tile[w * 32 + lane] = __funnelshift_l(raw[w + 1], raw[w], sh);
            }
            __syncwarp();
            for (;;) {
                // lane r: the cell r steps down the diagonal from (ti, tj), if the tile holds it
                const int ri = ti - lane, rj = tj - lane, wc = ((rj - 1) >> 3) - cw0;
                const bool held = ri >= 1 && rj >= 1 && ai - ri < 32 && wc >= 0;
                const int btr = held ? (int)((sm.tile[wc * 32 + (ai - ri)] >> (28 - 4 * ((rj - 1) & 7))) & 15u) : 3;
                const unsigned held0 = __ballot_sync(0xffffffffu, held) & 1u;
                if (!held0) break;                                      // the current cell is outside the tile (or the walk is over)
                // stored bits: 3 insertion opened (not an extension), 2 deletion opened, 1 insertion taken, 0 deletion
                // taken (it wins over the insertion); the reference's codes are move + "was an extension" flags
                const int b0 = __shfl_sync(0xffffffffu, btr, 0);
                if (state == 0 && (b0 & 3) == 0) {
                    // diagonal run: every leading lane whose cell also moves diagonally
                    const unsigned nd = __ballot_sync(0xffffffffu, !(held && (btr & 3) == 0));
                    const int run = nd ? __ffs((int)nd) - 1 : 32;
                    emit(0, run + ((raw_ops == 0 && strategy == kIgnore) ? seg : 0));
                    ti -= run; tj -= run; raw_ops += run;
                } else {
                    const int ins_ext = (b0 & 8) ? 0 : kInsertExt, del_ext = (b0 & 4) ? 0 : kDeleteExt;
                    // one move: inside a gap the state decides, otherwise the cell's own comparison results do
                    const bool in_ins = state == kInsertExt, in_del = state == kDeleteExt, fresh = !(in_ins || in_del);
                    const bool del = in_del || (fresh && (b0 & 1)), ins = !del && (in_ins || (b0 & 2));
                    ti -= ins ? 0 : 1; tj -= del ? 0 : 1;
                    state = del ? del_ext : ins ? ins_ext : 0;
                    raw_ops += fresh ? 1 : 0;
                    emit(del ? kDelete : kInsert, 1);
                }
            }
            __syncwarp();
        }
        {
            int off;
            if (strategy == kSoftClip) {
                if (tj > 0) emit(kStateClip, tj);
                off = ti;
            } else if (strategy == kIgnore) {
                if (tj > 0) emit(cur_state >= 0 ? cur_state : 0, tj);     // "same operation as the last one" (:391-394)
                off = ti - tj;
            } else {
                if (ti > 0) emit(kDelete, ti);
                else if (tj > 0) emit(kInsert, tj);
                off = 0;
            }
            if (cur_state >= 0) { if (lane == 0 && (uint32_t)n < a.cigar_cap) out[n] = make_int2(cur_len, cur_state); ++n; }
            if (lane == 0) {
                // forward order, appended to the batch's compact CIGAR array (what the host reads back: a few elements per
                // pair instead of cigar_cap); `out` was the scratch row of the backward pass
                const int stored = min(n, (int)a.cigar_cap);
                const uint32_t first = atomicAdd(a.compact_count, (uint32_t)stored);
                // (the compact array is sized from an estimate; when it runs over, the host sees the count and repeats the
                // batch with room for everything)
                if (first + (uint32_t)stored <= a.compact_cap)
                    for (int x = 0; x < stored; ++x) a.compact[first + x] = out[stored - 1 - x];
                a.compact_first[pd.index] = first;
                a.n_elem[pd.index] = n;
                a.offset[pd.index] = off;
                // the score of the cell the traceback starts from: INDEL always starts at (nrow, ncol), whatever the
                // end-cell search found (for IGNORE the walk may move to the last row; its score stays the search's)
                if (a.score) a.score[pd.index] = strategy == kIndel ? sm.lastcol[nrow] : best;
            }
        }
    }
}

}  // namespace

size_t smem_bytes_per_warp(uint32_t max_l1, uint32_t max_l2) { return per_warp_bytes(max_l1, max_l2); }

// Rows per lane for a matrix of l1 rows: as few blocks as the largest K allows, then the smallest instantiated K
// whose blocks hold the rows (the unused rows of the last lanes are computed and thrown away).
uint32_t pick_rows_per_lane(uint32_t l1)
{
    const uint32_t nblk = (l1 + 32 * kMaxRowsPerLane - 1) / (32 * kMaxRowsPerLane);
    const uint32_t per_block = (l1 + nblk - 1) / nblk;
    const uint32_t k = (per_block + 31) / 32;
    uint32_t best = kMaxRowsPerLane;
#define X(v) if (v >= k && v < best) best = v;
    SW_ROWS_PER_LANE(X)
#undef X
    return best;
}

template <bool CUTOFF>
static cudaError_t launch_align_t(const Args& a, int sm_count, cudaStream_t s, int* ctas_out)
{
    // Warps per CTA: four, fewer when the chunk's longest sequences make four warps' shared memory (~70 KB per warp at
    // 4 095 bases) exceed what a CTA may have.  The kernel carves shared memory by warp index and works with any count.
    int dev = 0, max_smem = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    if (e != cudaSuccess) return e;
    const size_t per_warp = smem_bytes_per_warp(a.max_l1, a.max_l2);
    int warps = kWarpsPerCta;
    while (warps > 1 && warps * per_warp > (size_t)max_smem) --warps;
    const size_t smem = warps * per_warp;
    auto kern = sw_align_kernel<CUTOFF>;
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int per_sm = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, warps * 32, smem);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) return cudaErrorInvalidConfiguration;
    const int want = (int)((a.npairs + warps - 1) / warps);
    const int ctas = want < sm_count * per_sm ? want : sm_count * per_sm;
    if (ctas_out) *ctas_out = ctas;
    kern<<<ctas, warps * 32, smem, s>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_align(const Args& a, int sm_count, cudaStream_t s, int* ctas_out)
{
    // The reference clamps the diagonal term at MATRIX_MIN_CUTOFF = -10^8 (PairWiseSW.h:31).  Every H is at least the
    // smallest boundary value plus min(i, j) diagonal steps, so with L = the longest sequence of the chunk no diagonal
    // term is below  min(0, open, open + (L-1) extend) + (L+1) min(match, mismatch, 0);  when that is above the cutoff the
    // clamp never acts and the kernel without it (one ALU instruction per cell fewer) gives identical results.
    const long long L = (long long)(a.max_l1 > a.max_l2 ? a.max_l1 : a.max_l2);
    long long bmin = 0;
    if ((long long)a.open < bmin) bmin = a.open;
    if ((long long)a.open + (L - 1) * a.extend < bmin) bmin = (long long)a.open + (L - 1) * a.extend;
    long long step = a.match < a.mismatch ? a.match : a.mismatch;
    if (step > 0) step = 0;
    const bool clamp_can_act = bmin + (L + 1) * step <= (long long)kMinCutoff;
    return clamp_can_act ? launch_align_t<true>(a, sm_count, s, ctas_out) : launch_align_t<false>(a, sm_count, s, ctas_out);
}

}  // namespace sw
