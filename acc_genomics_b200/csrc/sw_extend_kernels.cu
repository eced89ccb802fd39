// sw_extend_kernels.cu -- sm_100a BWA-MEM seed extension: ksw_extend2 of bwa 0.7.17, one warp per job.
//
// The recurrence, the band updates and every tie-break are those of bwa's ksw_extend2 (DESIGN.md section 14 restates it).
//
// Mapping to the machine:
//   * One warp extends one job; warps pull jobs (sorted largest first on the host) from an atomic cursor.
//   * Rows in sequence, columns across lanes.  An anti-diagonal wavefront like the aligner's does not fit: the band
//     [beg, end) of row i + 1 comes from a scan of all of row i, and an all-zero row or the Z-drop test ends the job after
//     a whole row.  So a row is processed left to right in chunks of 32 columns, lane k taking column j0 + k.
//   * The row array eh[0..qlen] of {H, E}, the query bytes and the m x m matrix live in the warp's shared memory; the row
//     loop reads global memory only for the target bytes (32 rows' worth per load).
//   * E is per column.  F is a warp scan: bwa computes E and F from M alone (never from H), so along a row
//         F(j) = max over beg <= k < j of (T_k - (j - 1 - k) e_ins),  T_k = max(M_k - o_ins - e_ins, 0),  F(beg) = 0,
//     an exclusive prefix maximum of T_k + k e_ins (five shuffles), shifted back by (j - 1) e_ins, with the maximum of
//     the columns left of the chunk carried from chunk to chunk.  F >= 0 for j > beg (T >= 0), so clamping at zero
//     turns the empty prefix into F(beg) = 0.
//   * eh[j].h receives H(i, j - 1): one shfl_up, and the carry from the chunk before (the first-column value for the
//     first chunk).  The row maximum is kept per lane (the last column of a lane's maximum) and reduced once per row:
//     the largest score, then the largest column holding it -- bwa's "the last column wins".
//   * The band update scans [beg, end] by ballots, 32 columns at a time, from each end.
//
// Ranges (all arithmetic is 32-bit; the host accepts only the domain of include/smithwaterman_cuda.h):
//   H, E, F are >= 0 (M may be negative, by at most 128), and a cell's H is h0 plus at most one matrix entry per row and
//   column visited: |H|, |E|, |F| <= 2^24 + 4095 * 127 < 2^26.  The first-column term o_del + e_del (i + 1) is at most
//   4096 + 4096 * 65535 < 2^28 + 2^12, and h0 minus it is above -2^29.  The Z-drop products ((i - max_i) - (mj - max_j))
//   e_del and the e_ins one: the row distance is at most 65536, the column distance at most 4096, so a product is at most
//   69632 * 4096 < 2^29, and max - m minus it stays within 2^30 of zero.  The scan values T_k + k e_ins are below
//   2^26 + 4095 * 4096 < 2^27; the empty-prefix value kNoScan = -2^29 minus (j - 1) e_ins (j < 4127) stays above -2^30.
#include "sw_extend_kernels.cuh"

namespace swx {
namespace {

constexpr unsigned kFull = 0xffffffffu;
constexpr int kNoScan = -(1 << 29);              // prefix maximum of no column (gives F = 0 after the clamp)

__host__ __device__ inline size_t query_bytes(uint32_t max_qlen) { return (max_qlen + 15) & ~(size_t)15; }

// eh ((max_qlen + 1) x 8 bytes), the query bytes, the matrix
__host__ __device__ inline size_t per_warp_bytes(uint32_t max_qlen)
{
    const size_t b = sizeof(int2) * (max_qlen + 1) + query_bytes(max_qlen) + kMaxAlphabet * kMaxAlphabet;
    return (b + 15) & ~(size_t)15;
}

__global__ void __launch_bounds__(kWarpsPerCta * 32) sw_extend_kernel(const __grid_constant__ Args a)
{
    extern __shared__ int4 smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    char* const base = reinterpret_cast<char*>(smem_raw) + warp * per_warp_bytes(a.max_qlen);
    int2* const eh = reinterpret_cast<int2*>(base);
    uint8_t* const qs = reinterpret_cast<uint8_t*>(eh + a.max_qlen + 1);
    int8_t* const mat = reinterpret_cast<int8_t*>(qs + query_bytes(a.max_qlen));
    const int m = a.m, o_del = a.o_del, e_del = a.e_del, o_ins = a.o_ins, e_ins = a.e_ins, zdrop = a.zdrop;
    const int oe_del = o_del + e_del, oe_ins = o_ins + e_ins;
    for (int x = lane; x < m * m; x += 32) mat[x] = a.mat[x];

    for (;;) {
        uint32_t p = 0;
        if (lane == 0) p = atomicAdd(a.counter, 1u);
        p = __shfl_sync(kFull, p, 0);
        if (p >= a.njobs) break;
        const JobDesc jd = a.jobs[p];
        const int qlen = (int)jd.q_len, tlen = (int)jd.t_len, h0 = jd.h0, w = jd.w;
        const uint8_t* const tg = a.target + jd.t_start;
        const uint8_t* const qg = a.query + jd.q_start;

        __syncwarp();                                   // the previous job's reads of eh and qs are done
        for (int j = lane; j < qlen; j += 32) qs[j] = qg[j];
        // first row: eh[1].h = max(h0 - o_ins - e_ins, 0), then down by e_ins while the previous is > e_ins, else 0
        const int h_first = h0 > oe_ins ? h0 - oe_ins : 0;
        for (int j = lane; j <= qlen; j += 32) eh[j] = make_int2(j == 0 ? h0 : max(h_first - (j - 1) * e_ins, 0), 0);
        __syncwarp();

        int beg = 0, end = qlen, best = h0, max_i = -1, max_j = -1, max_ie = -1, gscore = -1, max_off = 0;
        uint32_t cells = 0;
        int tword = 0;
        for (int i = 0; i < tlen; ++i) {
            if ((i & 31) == 0) tword = i + lane < tlen ? (int)tg[i + lane] : 0;
            const int8_t* const mrow = mat + __shfl_sync(kFull, tword, i & 31) * m;
            beg = max(beg, i - w);
            end = min(min(end, i + w + 1), qlen);
            int hcarry = beg == 0 ? max(h0 - (o_del + e_del * (i + 1)), 0) : 0;   // H(i, j0 - 1)
            int scarry = kNoScan;                                                  // max T_k + k e_ins, k < j0
            int mlane = 0, mjlane = -1;                                            // this lane's row maximum
            for (int j0 = beg; j0 < end; j0 += 32) {
                const int j = j0 + lane;
                const bool act = j < end;
                const int2 v = act ? eh[j] : make_int2(0, 0);
                const int M = v.x ? v.x + mrow[qs[j]] : 0;
                const int e = v.y;
                int S = act ? max(M - oe_ins, 0) + j * e_ins : kNoScan;
                #pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const int o = __shfl_up_sync(kFull, S, d);
                    if (lane >= d) S = max(S, o);
                }
                int ex = __shfl_up_sync(kFull, S, 1);
                ex = lane == 0 ? scarry : max(ex, scarry);
                scarry = max(scarry, __shfl_sync(kFull, S, 31));
                const int f = max(ex - (j - 1) * e_ins, 0);
                const int h = max(max(M, e), f);
                int hl = __shfl_up_sync(kFull, h, 1);
                if (lane == 0) hl = hcarry;
                if (act) {
                    eh[j] = make_int2(hl, max(e - e_del, max(M - oe_del, 0)));
                    if (h >= mlane) { mlane = h; mjlane = j; }
                }
                hcarry = __shfl_sync(kFull, h, min(31, end - 1 - j0));
            }
            cells += (uint32_t)max(end - beg, 0);
            if (lane == 0) eh[end] = make_int2(hcarry, 0);
            if (max(beg, end) == qlen) {                // the row reached the end of the query
                max_ie = gscore > hcarry ? max_ie : i;
                gscore = max(gscore, hcarry);
            }
            const int mrow_max = __reduce_max_sync(kFull, mlane);
            if (mrow_max == 0) break;
            const int mj = __reduce_max_sync(kFull, mlane == mrow_max ? mjlane : -1);
            if (mrow_max > best) {
                best = mrow_max; max_i = i; max_j = mj;
                max_off = max(max_off, abs(mj - i));
            } else if (zdrop > 0) {
                if (i - max_i > mj - max_j) {
                    if (best - mrow_max - ((i - max_i) - (mj - max_j)) * e_del > zdrop) break;
                } else {
                    if (best - mrow_max - ((mj - max_j) - (i - max_i)) * e_ins > zdrop) break;
                }
            }
            __syncwarp();
            // band of the next row: first non-zero entry in [beg, end), last one in [beg, end]
            int nb = end;
            for (int j0 = beg; j0 < end; j0 += 32) {
                const int j = j0 + lane;
                const int2 v = j < end ? eh[j] : make_int2(0, 0);
                const unsigned b = __ballot_sync(kFull, (v.x | v.y) != 0);
                if (b) { nb = j0 + __ffs((int)b) - 1; break; }
            }
            beg = nb;
            int ne = beg - 1;
            for (int j1 = end; j1 >= beg; j1 -= 32) {
                const int j = j1 - lane;
                const int2 v = j >= beg ? eh[j] : make_int2(0, 0);
                const unsigned b = __ballot_sync(kFull, (v.x | v.y) != 0);
                if (b) { ne = j1 - (__ffs((int)b) - 1); break; }
            }
            end = min(ne + 2, qlen);
            __syncwarp();                               // the scans' reads before the next row's writes
        }
        if (lane == 0) {
            int32_t* o = a.out + 6 * (size_t)jd.index;
            o[0] = best; o[1] = max_j + 1; o[2] = max_i + 1; o[3] = max_ie + 1; o[4] = gscore; o[5] = max_off;
            atomicAdd(a.cells, (unsigned long long)cells);
        }
    }
}

}  // namespace

cudaError_t launch_extend(const Args& a, int sm_count, cudaStream_t s)
{
    int dev = 0, max_smem = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    if (e != cudaSuccess) return e;
    const size_t per_warp = per_warp_bytes(a.max_qlen);
    int warps = kWarpsPerCta;
    while (warps > 1 && warps * per_warp > (size_t)max_smem) --warps;
    const size_t smem = warps * per_warp;
    e = cudaFuncSetAttribute(sw_extend_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int per_sm = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sw_extend_kernel, warps * 32, smem);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) return cudaErrorInvalidConfiguration;
    const long long want = ((long long)a.njobs + warps - 1) / warps;
    const int ctas = (int)(want < (long long)sm_count * per_sm ? want : (long long)sm_count * per_sm);
    sw_extend_kernel<<<ctas, warps * 32, smem, s>>>(a);
    return cudaGetLastError();
}

}  // namespace swx
