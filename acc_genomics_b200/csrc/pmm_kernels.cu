// pmm_kernels.cu -- sm_100a kernels of the PairHMM forward path.
//
// The recurrence and its operation order are those of the reference's AVX implementation
// (/root/reference/pairhmm/xlnx/host/avx-pairhmm-template.h:183-198 computeMXY, :136-177 boundary conditions,
// :308-343 reduction); SURVEY.md appendix A restates them.  Every multiply and add below is an individually
// rounded __fmul_rn/__fadd_rn (never contracted), the file is compiled with -ftz=true, and the tables come from
// the host libm, so the float result is bit-identical to the reference built without FMA contraction.
//
// Mapping to the machine (B200-first, not a translation of the AVX or FPGA code):
//   * One read occupies W lanes of a warp (W = 8, 16 or 32); each lane keeps K consecutive rows of the M/X/Y
//     matrices and their transition parameters in registers.  Rows are end-aligned: the read's last row is row
//     K-1 of lane W-1, the unused rows at the top are "boundary rows" (M = X = 0, Y = 2^120/haplen), which also
//     absorb the undefined value lane 0 receives from the shuffle.
//   * The anti-diagonal wavefront runs across lanes: at step t lane l works on column t - l.  The last row of
//     lane l-1 reaches lane l through three __shfl_up_sync per step (M, X, Y), i.e. 3/K shuffles per cell.
//   * A warp does not handle one pair at a time: the haplotypes of a region are concatenated into one stream
//     with separator elements, and the wavefront flows from one haplotype straight into the next, so the
//     fill/drain bubble (W-1 steps) is paid once per task instead of once per pair.  A separator step resets the
//     lane's state and (in lane W-1) stores the previous haplotype's result.
//   * The match/mismatch emission weight is not selected per cell (that would cost a LOP3 + FSEL issue slot each;
//     the measured issue rate is 1 instr/clk/SMSP for FP32 and ALU alike, tools/microbench/issue_mix2.cu): each
//     warp stages a [5 classes][K rows] weight table for its reads in shared memory, laid out so that one
//     LDS.128 per 4 rows fetches the weights for whatever haplotype base the lane is looking at (16 bytes per lane,
//     consecutive lanes consecutive: the 512 bytes of a warp take the minimum of four wavefronts).
//   * Steady-state steps are branch-free; only the W steps around a separator run the checked variant.
//   * The AVX code's stripe initialisation feeds M[r-1][1] into Y[r][1] for the first row of every 8-row stripe
//     (avx-pairhmm-template.h:171-176); that value is exactly 0 for r >= 3, so there is nothing to reproduce.
//   * Work is pulled by warps from a global queue (atomicAdd), grid = SMs x resident CTAs.
#include "pmm_kernels.cuh"

#include <algorithm>
#include <atomic>
#include <cfloat>
#include <type_traits>

namespace pmm {
namespace {

constexpr int kSteadyUnrollF32 = 4;            // steps per trip of the branch-free loop
// the double kernel is bound by the latency of its dependent DP chains, not by issue slots: a longer trip gives ptxas
// more independent work to put between them (measured on config 3: 2 steps 2.36 ms, 4 steps 2.30, 8 steps 2.28)
constexpr int kSteadyUnrollF64 = 8;

__device__ __forceinline__ int base_class(unsigned ch)
{
    // A,C,T,G,N -> 0..4, everything else 0 (ConvertChar's zero-initialised table, host_type.h:123-143)
    return ch == 'C' ? 1 : ch == 'T' ? 2 : ch == 'G' ? 3 : ch == 'N' ? 4 : 0;
}

template <typename T> struct Arith;

template <> struct Arith<float> {
    static constexpr int kVec = 4;             // elements per 16-byte shared-memory access
    static __device__ __forceinline__ float mul(float a, float b) { return __fmul_rn(a, b); }
    static __device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
    static __device__ __forceinline__ float sub(float a, float b) { return __fsub_rn(a, b); }
    static __device__ __forceinline__ float div(float a, float b) { return __fdiv_rn(a, b); }
    static __device__ __forceinline__ float ph2pr(const DeviceTables& t, int q) { return __ldg(t.ph2pr_f + q); }
    static __device__ __forceinline__ float m2m(const DeviceTables& t, int i) { return __ldg(t.m2m_f + i); }
};

template <> struct Arith<double> {
    static constexpr int kVec = 2;
    static __device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
    static __device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
    static __device__ __forceinline__ double sub(double a, double b) { return __dsub_rn(a, b); }
    static __device__ __forceinline__ double div(double a, double b) { return __ddiv_rn(a, b); }
    static __device__ __forceinline__ double ph2pr(const DeviceTables& t, int q) { return __ldg(t.ph2pr_d + q); }
    static __device__ __forceinline__ double m2m(const DeviceTables& t, int i) { return __ldg(t.m2m_d + i); }
};

// x86 flush-to-zero for doubles: a product below DBL_MIN becomes +0 (all operands here are non-negative).
// Sums of flushed, non-negative operands can never be subnormal, so only products need it.
template <bool FLUSH> __device__ __forceinline__ double flush(double x)
{
    if (FLUSH) return x < DBL_MIN ? 0.0 : x;
    return x;
}
template <bool FLUSH> __device__ __forceinline__ float flush(float x) { return x; }   // -ftz=true does it in hardware

template <typename T> __device__ __forceinline__ T ld_cg(const T* p) { return __ldcg(p); }

template <typename T, int K>
__host__ __device__ constexpr int wtab_elems() { return 5 * ((K + Arith<T>::kVec - 1) / Arith<T>::kVec) * 32 * Arith<T>::kVec; }

// ---------------------------------------------------------------------------------------------------------
// The forward kernel.
// ---------------------------------------------------------------------------------------------------------
// ---- fallback count: the float pass counts the pairs whose result is below 1e-28f the moment the result exists ----
// (Tried and measured on B200, see DESIGN.md section 4.5: *consuming* a fallback list inside the float kernel, so that the
// double re-run overlaps the float pass, is slower than a separate double launch -- the two loop bodies evict each
// other from the instruction caches and the double tasks run at the float kernel's lower occupancy.)
__device__ __forceinline__ void count_fallback(const FallbackQueue& fq)
{
    // The pair itself is found again by fallback_scan_kernel's scan of the results (which groups the failing pairs of
    // a read into one task); the float pass only keeps the total, which sizes those tasks.
    atomicAdd(fq.reserve, 1u);
}

// Fast mode: a result too close to 1e-28f to trust the decision.  The re-check task writes the exact float result
// over the fast one (out_base = the pair's own result index) and, being an exact kernel with kPush, counts the
// pair as a fallback if that is what the reference would do.
__device__ __forceinline__ void push_recheck(const FallbackQueue& fq, uint32_t read, uint32_t hap, uint32_t out_index)
{
    const uint32_t slot = atomicAdd(fq.recheck_count, 1u);
    if (slot >= fq.capacity) return;
    Task t;
    t.read[0] = read; t.read[1] = t.read[2] = t.read[3] = 0;
    t.out_base[0] = out_index; t.out_base[1] = t.out_base[2] = t.out_base[3] = 0;
    t.hap_first = hap; t.nhaps = 1; t.nreads = 1; t.param_off = 0;
    fq.recheck_tasks[slot] = t;
}

// ---------------------------------------------------------------------------------------------------------
// One warp-task: the reads of one group against a run of haplotypes.
// ---------------------------------------------------------------------------------------------------------
// F: bit flags.  kFlush: emulate x86 flush-to-zero after every double product.  kPush: append results below the
// fallback threshold to the fallback list (float).  kFast: the float cell update contracted to 8 instructions (FADD +
// 4 FMUL + 3 FFMA; results within a few ulp of the exact order; the engine re-checks everything near the threshold with
// an exact kernel).
// kInline: compute the float row parameters in the kernel instead of reading read_params_kernel's planes (single-pair
// re-check tasks have no parameter block).
constexpr int kFlush = 1, kPush = 2, kFast = 4, kInline = 8;
// kRetry (kernel level, double only): a pair whose result is below tiny_threshold is run again at once with
// kFlush -- the case where x86 flush-to-zero of intermediate products may have changed the reference's result.
constexpr int kRetry = 16;
// kList (double re-run): the task's haplotypes are not a run of consecutive ones but entries hap_first .. hap_first +
// nhaps - 1 of a.hap_list (the failing haplotypes of one read, fallback_scan_kernel).  The wavefront still flows from
// one haplotype into the next; a lane re-points its stream pointer when it crosses a separator.
constexpr int kList = 32;

// A row's entries in the five class tables of a lane's weight table (w: the row's entry of class 0): the match weight
// where the haplotype class equals the read's base class or either is N (class 4), the mismatch weight elsewhere.
template <typename T, int CLS_STRIDE>
__device__ __forceinline__ void scatter_weights(T* w, unsigned cls, T mw, T xw)
{
    #pragma unroll
    for (int h = 0; h < 5; ++h) {
        const bool match = (cls == (unsigned)h) || cls == 4 || h == 4;
        w[h * CLS_STRIDE] = match ? mw : xw;
    }
}

template <typename T, int K, int W, bool STRIPED, int F>
__device__ __forceinline__ void run_task(const ForwardArgs& a, const Task* tk, T* wtab, const int lane,
                                         const uint32_t gwarp, const FallbackQueue& fq)
{
    using A = Arith<T>;
    constexpr bool FLUSH = (F & kFlush) != 0, PUSH = (F & kPush) != 0, FAST = (F & kFast) != 0, INLINE = (F & kInline) != 0;
    constexpr bool LIST = (F & kList) != 0;
    constexpr bool kIsFloat = std::is_same<T, float>::value;
    static_assert(kIsFloat || !(FAST || PUSH || INLINE), "float-only flags");
    constexpr int VEC = A::kVec;
    constexpr int KQ = (K + VEC - 1) / VEC;           // 16-byte weight vectors per lane and class
    constexpr int CLS_STRIDE = KQ * 32 * VEC;         // elements between the tables of two haplotype classes
    static_assert(W == 8 || W == 16 || W == 32, "W");
    static_assert(!STRIPED || W == 32, "striped variant handles one read per warp");
    const int g = lane / W, l = lane % W;
    T* wlane = wtab + lane * VEC;
    const T* inity = static_cast<const T*>(a.inity);
    T* out = static_cast<T*>(a.out);

    const uint32_t hap_first = tk->hap_first, nhaps = tk->nhaps;
    const bool valid = (uint32_t)g < tk->nreads;
    ReadDesc rd = {0u, 0u, 0u};
    uint32_t out_base = 0;
    if (valid) { rd = a.reads[tk->read[g]]; out_base = tk->out_base[g]; }
    const int R = (int)rd.len;
    const int nstripes = STRIPED ? (R + W * K) / (W * K) : 1;       // ceil((R + 1) / (W*K))
    const int pad = nstripes * W * K - R;                            // >= 1 boundary rows at the top

    // haplotype n of the task, as an index into spos / inity
    auto hap_at = [&](uint32_t n) -> uint32_t { return LIST ? __ldg(a.hap_list + hap_first + n) : hap_first + n; };
    const uint32_t s0 = a.spos[hap_at(0)];
    int Lc;                                                          // elements incl. the terminal separator
    if constexpr (LIST) {
        // the task's haplotypes lie anywhere in the stream: add up their lengths (+ one separator each)
        static_assert(!LIST || W == 32, "list tasks: one read per warp");
        uint32_t len = 0;
        for (uint32_t n = lane; n < nhaps; n += 32) { const uint32_t h = hap_at(n); len += a.spos[h + 1] - a.spos[h]; }
        #pragma unroll
        for (int o = 16; o; o >>= 1) len += __shfl_xor_sync(0xffffffffu, len, o);
        Lc = (int)len + 1;
    } else {
        Lc = (int)(a.spos[hap_first + nhaps] - s0) + 1;
    }
    const int Tsteps = Lc + W - 1;

    T* scM = nullptr; T* scX = nullptr; T* scY = nullptr;
    if (STRIPED) {
        scM = static_cast<T*>(a.scratch) + (size_t)gwarp * 3 * a.scratch_stride;
        scX = scM + a.scratch_stride; scY = scX + a.scratch_stride;
    }

    #pragma unroll 1
    for (int stripe = 0; stripe < nstripes; ++stripe) {
        const uint8_t* sp = a.stream + s0 - l;                       // this lane's element at step t is sp[t]
        // ---- per-row parameters (avx-pairhmm-template.h:108-127, :155-158) --------------------------
        T pMM[K], pG[K], pMX[K], pMY[K], pC[K];       // pXX == pYY == ph2pr[c] (:119-121)
        T pX0 = (T)0;                                                // pC[0] as the X update of row 0 sees it
        unsigned padmask = 0;
        __syncwarp();                                                // previous task / stripe done with wtab
        if constexpr (kIsFloat && !INLINE) {
            // float pass: the rows were prepared once per read by read_params_kernel; W consecutive lanes read
            // consecutive floats, all 8K loads are independent
            constexpr int KW = K * W;
            const float* pb = a.params + tk->param_off + ((size_t)(STRIPED ? 0 : g) * nstripes + stripe) * (kParamPlanes * KW) + l;
            #pragma unroll
            for (int j = 0; j < K; ++j) {
                const float* pj = pb + j * W;
                pMM[j] = __ldg(pj + 0 * KW); pG[j] = __ldg(pj + 1 * KW); pMX[j] = __ldg(pj + 2 * KW);
                pMY[j] = __ldg(pj + 3 * KW); pC[j] = __ldg(pj + 4 * KW);
                const float mw = __ldg(pj + 5 * KW), xw = __ldg(pj + 6 * KW);
                const unsigned cls = __float_as_uint(__ldg(pj + 7 * KW));
                if (cls == kPadClass) padmask |= 1u << j;
                if (j == 0) pX0 = cls == kPadClass ? 0.0f : pC[0];
                scatter_weights<T, CLS_STRIDE>(wlane + (j / VEC) * 32 * VEC + (j % VEC), cls, mw, xw);
            }
        } else {
            #pragma unroll
            for (int j = 0; j < K; ++j) {
                const int r0 = stripe * W * K + l * K + j - pad;          // 0-based read base of this row
                T mw = (T)0, xw = (T)0;
                int cls = 0;
                if (r0 >= 0 && valid) {
                    // the same derivation as read_params_kernel's (kept in two places: as one helper it changes the
                    // SASS of the double kernels or of read_params_kernel)
                    const uint8_t* b = a.read_blob + rd.off + r0;
                    cls = base_class(b[0]);
                    const int q_ = b[rd.stride] & 127, i_ = b[2 * rd.stride] & 127;
                    const int d_ = b[3 * rd.stride] & 127, c_ = b[4 * rd.stride] & 127;
                    const int mx = max(i_, d_), mn = min(i_, d_);
                    pMM[j] = A::m2m(a.tab, ((mx * (mx + 1)) >> 1) + mn);
                    const T pc = A::ph2pr(a.tab, c_);
                    pG[j] = A::sub((T)1.0, pc);
                    pMX[j] = A::ph2pr(a.tab, i_);
                    pMY[j] = A::ph2pr(a.tab, d_);
                    pC[j] = pc;
                    if (j == 0) pX0 = pc;
                    const T dm = A::ph2pr(a.tab, q_);
                    mw = A::sub((T)1.0, dm);
                    xw = A::div(dm, (T)3.0);
                } else {
                    // boundary row: M = 0, Y keeps its value, X copies the row above; a boundary row 0 ignores the
                    // row above (pX0 = 0: whatever the shuffle delivers, lane 0's own value included) so X stays 0
                    pMM[j] = (T)0; pG[j] = (T)0; pMX[j] = (T)0; pMY[j] = (T)0; pC[j] = (T)1.0;
                    padmask |= 1u << j;
                }
                scatter_weights<T, CLS_STRIDE>(wlane + (j / VEC) * 32 * VEC + (j % VEC), (unsigned)cls, mw, xw);
            }
        }
        __syncwarp();

        T M[K], X[K], Y[K];
        #pragma unroll
        for (int j = 0; j < K; ++j) { M[j] = (T)0; X[j] = (T)0; Y[j] = (T)0; }
        T dM = (T)0, dX = (T)0, dY = (T)0;        // last row of the lane above, previous column (diagonal)
        T sM = (T)0, sX = (T)0;                   // running sums of the read's last row
        int nsep = 0;
        bool done = false;
        const bool last_stripe = stripe == nstripes - 1;
        const bool carry_in = STRIPED && stripe > 0 && l == 0;
        const bool carry_out = STRIPED && !last_stripe && l == W - 1;

        // One column of K cells.  inM/inX/inY: last row of the lane above at this column.
        auto cells = [&](unsigned e, T inM, T inX, T inY) {
            const T* wp = wlane + e * CLS_STRIDE;
            T w[KQ * VEC];
            #pragma unroll
            for (int m = 0; m < KQ; ++m) {
                if (VEC == 4) {
                    const float4 v = *reinterpret_cast<const float4*>(wp + m * 32 * VEC);
                    w[m * VEC + 0] = v.x; w[m * VEC + 1] = v.y; w[m * VEC + 2] = v.z; w[m * VEC + 3] = v.w;
                } else {
                    const double2 v = *reinterpret_cast<const double2*>(wp + m * 32 * VEC);
                    w[m * VEC + 0] = v.x; w[m * VEC + 1] = v.y;
                }
            }
            T Mn[K], Xn[K], Yn[K];
            #pragma unroll
            for (int j = K - 1; j >= 0; --j) {
                const T md = j ? M[j - 1] : dM, xd = j ? X[j - 1] : dX, yd = j ? Y[j - 1] : dY;
                if constexpr (FAST) {
                    // 8 instructions per cell instead of 12: M = fma(Xd + Yd, pG, Md pMM) w, and FMUL + FFMA for each of X
                    // and Y.  What counts beside the instructions is their register operands -- the register file feeds
                    // two per issue slot, a three-register FFMA costs ~1.5 slots (tools/microbench/ffma_regs.cu) -- 19
                    // here against 24 in the exact order.  (Tried: folding w into pre-multiplied pMM w / pG w tables,
                    // 7 instructions and 17 operands, needs a second LDS.128 per four rows and saturates the
                    // shared-memory pipe: 2.74 against 2.92 TCUPS on config 2.)
                    Mn[j] = __fmul_rn(__fmaf_rn(__fadd_rn(xd, yd), pG[j], __fmul_rn(md, pMM[j])), w[j]);
                    Yn[j] = __fmaf_rn(Y[j], pC[j], __fmul_rn(M[j], pMY[j]));
                } else {
                    // M = ((Md*pMM + Xd*pGAPM) + Yd*pGAPM) * w        (avx-pairhmm-template.h:188)
                    const T t3 = A::add(flush<FLUSH>(A::mul(md, pMM[j])), flush<FLUSH>(A::mul(xd, pG[j])));
                    const T t5 = A::add(t3, flush<FLUSH>(A::mul(yd, pG[j])));
                    Mn[j] = flush<FLUSH>(A::mul(t5, w[j]));
                    // Y = Mleft*pMY + Yleft*pYY                        (:197)
                    Yn[j] = A::add(flush<FLUSH>(A::mul(M[j], pMY[j])), flush<FLUSH>(A::mul(Y[j], pC[j])));
                }
            }
            #pragma unroll
            for (int j = 0; j < K; ++j) {
                const T mu = j ? Mn[j - 1] : inM, xu = j ? Xn[j - 1] : inX;
                // X = Mup*pMX + Xup*pXX                             (:194)
                if constexpr (FAST) Xn[j] = __fmaf_rn(xu, j ? pC[j] : pX0, __fmul_rn(mu, pMX[j]));
                else Xn[j] = A::add(flush<FLUSH>(A::mul(mu, pMX[j])), flush<FLUSH>(A::mul(xu, j ? pC[j] : pX0)));
            }
            #pragma unroll
            for (int j = 0; j < K; ++j) { M[j] = Mn[j]; X[j] = Xn[j]; Y[j] = Yn[j]; }
            sM = A::add(sM, M[K - 1]);          // (:328,:331) two sums, left to right
            sX = A::add(sX, X[K - 1]);
            dM = inM; dX = inX; dY = inY;
        };

        // What a lane needs when it crosses the separator in front of haplotype hn -- its initial Y value and, for list
        // tasks, where its bases are and the first of them.  The same for every lane, so it is loaded once per window
        // and a whole haplotype ahead (fetch_hap below), not by each lane in the middle of its separator step where a
        // chain of dependent loads would stall the warp 32 times per haplotype.
        uint32_t hn = 0;                      // index (within the task) of the next separator lane 0 will meet
        T w_iy = (T)0;
        uint32_t w_ps = 0, w_len = 0;
        unsigned w_first = 0;
        auto fetch_hap = [&](uint32_t n) {
            w_iy = (T)0; w_len = 0; w_first = 0;
            if (n < nhaps) {
                const uint32_t h = hap_at(n);
                w_iy = inity[h];
                if constexpr (LIST) { w_ps = a.spos[h]; w_len = a.spos[h + 1] - w_ps; w_first = a.stream[w_ps + 1]; }
            }
        };

        // Step with every check: separators, fill/drain, stripe carries.
        auto checked_step = [&](int t, unsigned e) -> bool {
            bool repointed = false;
            T inM = __shfl_up_sync(0xffffffffu, M[K - 1], 1, W);
            T inX = __shfl_up_sync(0xffffffffu, X[K - 1], 1, W);
            T inY = __shfl_up_sync(0xffffffffu, Y[K - 1], 1, W);
            const int p = t - l;
            const bool active = p >= 0 && !done;
            if (carry_in && active) { inM = ld_cg(scM + p); inX = ld_cg(scX + p); inY = ld_cg(scY + p); }
            if (active) {
                if (e == kSep) {
                    if (nsep > 0 && l == W - 1 && valid && last_stripe) {
                            const T res = A::add(sM, sX);
                            out[out_base + nsep - 1] = res;
                            if constexpr (PUSH) {
                                // exact kernels: lo == hi == 1e-28f, the reference's test, a float compare
                                // (PairHMMWorker.cpp:176; NaN -> false).  Fast kernels: results in [lo, hi) are too close
                                // to the threshold to decide and go to the exact re-check list instead.
                                if (res < fq.hi) {
                                    if (res < fq.lo) count_fallback(fq);
                                    else push_recheck(fq, tk->read[g], hap_first + nsep - 1, out_base + nsep - 1);
                                }
                            }
                        }
                    done = nsep == (int)nhaps;
                    T iy = (T)0;
                    if (!done) {
                        // this separator stands at step t for this lane; from here on a list task's lane reads the
                        // haplotype that starts here
                        if (nsep == (int)hn) {
                            iy = w_iy;
                            if constexpr (LIST) sp = a.stream + w_ps - t;
                        } else {
                            // a haplotype shorter than the warp: this lane crosses a second separator inside the window
                            const uint32_t h = hap_at((uint32_t)nsep);
                            iy = inity[h];
                            if constexpr (LIST) sp = a.stream + a.spos[h] - t;
                        }
                        repointed = LIST;
                    }
                    ++nsep;
                    #pragma unroll
                    for (int j = 0; j < K; ++j) { M[j] = (T)0; X[j] = (T)0; Y[j] = (padmask >> j) & 1 ? iy : (T)0; }
                    sM = (T)0; sX = (T)0;
                    dM = inM; dX = inX; dY = inY;
                } else {
                    cells(e, inM, inX, inY);
                }
                if (carry_out) { scM[p] = M[K - 1]; scX[p] = X[K - 1]; scY[p] = Y[K - 1]; }
            }
            return repointed;
        };

        // Branch-free step: every lane is inside the bases of a haplotype.
        auto steady_step = [&](int t, unsigned e) {
            T inM = __shfl_up_sync(0xffffffffu, M[K - 1], 1, W);
            T inX = __shfl_up_sync(0xffffffffu, X[K - 1], 1, W);
            T inY = __shfl_up_sync(0xffffffffu, Y[K - 1], 1, W);
            if (STRIPED) {
                const int p = t - l;
                if (carry_in) { inM = ld_cg(scM + p); inX = ld_cg(scX + p); inY = ld_cg(scY + p); }
                cells(e, inM, inX, inY);
                if (carry_out) { scM[p] = M[K - 1]; scX[p] = X[K - 1]; scY[p] = Y[K - 1]; }
            } else {
                cells(e, inM, inX, inY);
            }
        };

        int t = 0;
        int next_sep = 0;                     // step at which lane 0 meets separator hn
        unsigned e = sp[0];
        fetch_hap(0);
        while (t < Tsteps) {
            // checked window: lane l meets the separator at step next_sep + l
            int wend = next_sep + W;
            if (wend > Tsteps) wend = Tsteps;
            if constexpr (LIST) {
                for (; t < wend; ++t) {
                    const unsigned en = sp[t + 1];
                    // a lane that re-pointed reads the first base of its new haplotype next, not what follows the
                    // separator in memory
                    if (checked_step(t, e)) e = nsep - 1 == (int)hn ? w_first : sp[t + 1];
                    else e = en;
                }
                ++hn;
                next_sep = hn <= nhaps ? next_sep + (int)w_len : Tsteps + W;
            } else {
                for (; t < wend; ++t) {
                    const unsigned en = sp[t + 1];
                    checked_step(t, e);
                    e = en;
                }
                ++hn;
                next_sep = hn <= nhaps ? (int)(a.spos[hap_first + hn] - s0) : Tsteps + W;
            }
            fetch_hap(hn);                    // for the next window, a whole haplotype from now
            int send = next_sep < Tsteps ? next_sep : Tsteps;
            // kSteadyUnroll steps per trip: the element loads use one pointer with immediate offsets
            constexpr int kSteadyUnroll = kIsFloat ? kSteadyUnrollF32 : kSteadyUnrollF64;
            const uint8_t* q = sp + t;
            #pragma unroll 1
            for (; t + kSteadyUnroll <= send; t += kSteadyUnroll, q += kSteadyUnroll) {
                unsigned en[kSteadyUnroll];
                #pragma unroll
                for (int u = 0; u < kSteadyUnroll; ++u) en[u] = q[u + 1];
                steady_step(t, e);
                #pragma unroll
                for (int u = 1; u < kSteadyUnroll; ++u) steady_step(t + u, en[u - 1]);
                e = en[kSteadyUnroll - 1];
            }
            #pragma unroll 1
            for (; t < send; ++t) {
                const unsigned en = sp[t + 1];
                steady_step(t, e);
                e = en;
            }
        }
    }
}

template <typename T, int K, int W, bool STRIPED, int F>
__global__ void __launch_bounds__(kWarpsPerCta * 32, resident_ctas<T>(K)) pmm_forward_kernel(const ForwardArgs a, const FallbackQueue fq)
{
    extern __shared__ uint4 smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    T* wtab = reinterpret_cast<T*>(smem_raw) + warp * wtab_elems<T, K>();
    const uint32_t ntasks = a.ntasks_dev ? *a.ntasks_dev : a.ntasks;
    const uint32_t gwarp = blockIdx.x * kWarpsPerCta + warp;
    for (;;) {
        uint32_t ti = 0;
        if (lane == 0) ti = atomicAdd(a.counter, 1u);
        ti = __shfl_sync(0xffffffffu, ti, 0);
        if (ti >= ntasks) break;
        run_task<T, K, W, STRIPED, F & ~kRetry>(a, a.tasks + ti, wtab, lane, gwarp, fq);
        if constexpr ((F & kRetry) != 0) {
            // Intermediate products below DBL_MIN are flushed to zero on the reference's x86 (FTZ on); they can only
            // influence results that are themselves tiny.  Everything below tiny_threshold (2^-800, scaled by 2^1020) is
            // recomputed, one pair at a time, with the flush emulated after every product; above it the two
            // arithmetics agree.
            static_assert(std::is_same<T, double>::value && W == 32, "retry is for the one-read double tasks");
            __syncwarp();
            const Task tk = a.tasks[ti];
            for (uint32_t n0 = 0; n0 < tk.nhaps; n0 += 32) {
                double r = 1.0;                                                      // written by lane 31 a moment ago
                if (n0 + lane < tk.nhaps) r = __ldcg(static_cast<const double*>(a.out) + tk.out_base[0] + n0 + lane);
                unsigned m = __ballot_sync(0xffffffffu, r < a.tiny_threshold);
                while (m) {
                    const uint32_t n = n0 + (uint32_t)__ffs(m) - 1;
                    m &= m - 1;
                    Task one = tk;
                    one.hap_first = tk.hap_first + n; one.nhaps = 1; one.out_base[0] = tk.out_base[0] + n;
                    if (lane == 0) atomicAdd(a.tiny_count, 1u);
                    run_task<T, K, W, STRIPED, (F & ~kRetry) | kFlush>(a, &one, wtab, lane, gwarp, fq);
                }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// Fallback tasks of the double re-run: one warp per result row (one read against the haplotypes of its region).
// ---------------------------------------------------------------------------------------------------------
// The reference re-runs every pair with raw < 1e-28f in double, one pair at a time (PairHMMWorker.cpp:176-184).  Here
// the failing haplotypes of a read become tasks of `run` haplotypes each, so that the wavefront bubble, the row
// parameters (a double division per row) and the shared-memory weight table are paid once per task, not once per
// pair.  `run` follows from the number of failing pairs the float pass counted: enough tasks to keep every resident
// warp of the double kernel supplied, never more than max_run.  Slot k of the fallback list (out_index[k], hap_list[k],
// and the double result the kernel writes to dres[k]) belongs to one pair; a task owns consecutive slots.
// Two launches: the scan finds the failing pairs, fills the slots and counts the tasks per cost class; the second
// writes the tasks longest first (a counting sort on kCostClasses classes), because warps pull tasks in order and the
// double pass of a typical job is only two or three tasks deep per warp -- its tail is what the order decides
// (measured on config 2: 0.31 ms longest-first, 0.38 ms in row order).
struct RowCut { uint32_t run, ntask; };

__device__ __forceinline__ uint32_t fallback_run_cap(const FallbackBuild& b, uint32_t total)
{
    return max(1u, min(b.max_run, total / max(1u, b.target_tasks)));
}
// reads longer than one stripe of the double kernel carry rows through scratch sized for one haplotype: one pair per task
__device__ __forceinline__ RowCut cut_row(const FallbackBuild& b, uint32_t read, uint32_t n, uint32_t run_cap)
{
    const uint32_t run = b.reads[read].len + 1 > b.single_stripe_rows ? 1u : run_cap;
    return RowCut{run, (n + run - 1) / run};
}
// wavefront steps of task t of a row (haplotype bases + one separator each) and its cost class, 0 = the longest
__device__ __forceinline__ uint32_t task_class(const FallbackBuild& b, uint32_t slot, uint32_t n, uint32_t ntask, uint32_t t, uint32_t run_cap)
{
    const uint32_t k0 = (uint32_t)((uint64_t)n * t / ntask), k1 = (uint32_t)((uint64_t)n * (t + 1) / ntask);
    uint32_t cost = 0;
    for (uint32_t k = k0; k < k1; ++k) { const uint32_t h = b.hap_list[slot + k]; cost += b.spos[h + 1] - b.spos[h]; }
    const uint32_t cmax = run_cap * (b.max_hap_len + 1);
    return (kCostClasses - 1) - min((uint32_t)(kCostClasses - 1), (uint32_t)((uint64_t)cost * (kCostClasses - 1) / cmax));
}

__device__ __forceinline__ void row_of(const FallbackBuild& b, uint32_t row, RegionDesc& rg, uint32_t& read, uint32_t& base)
{
    uint32_t lo = 0, hi = b.num_region;                       // last region with row_first <= row
    while (hi - lo > 1) { const uint32_t mid = (lo + hi) >> 1; if (b.regions[mid].row_first <= row) lo = mid; else hi = mid; }
    rg = b.regions[lo];
    const uint32_t r = row - rg.row_first;
    read = rg.read_first + r; base = rg.out_first + r * rg.nhaps;
}

__global__ void __launch_bounds__(256) fallback_scan_kernel(const FallbackBuild b)
{
    const uint32_t total = b.ctrl[0];
    if (total == 0) return;
    const uint32_t run_cap = fallback_run_cap(b, total);
    const uint32_t lane = threadIdx.x & 31, warps = (gridDim.x * blockDim.x) >> 5;
    const unsigned lt = (1u << lane) - 1u;
    for (uint32_t row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; row < b.num_rows; row += warps) {
        RegionDesc rg; uint32_t read, base;
        row_of(b, row, rg, read, base);
        const float* raw = b.raw + base;
        uint32_t n = 0;
        for (uint32_t h0 = 0; h0 < rg.nhaps; h0 += 32) {
            const bool fail = h0 + lane < rg.nhaps && raw[h0 + lane] < b.threshold;      // NaN -> false, like the reference
            n += __popc(__ballot_sync(0xffffffffu, fail));
        }
        uint32_t slot = 0;
        if (n && lane == 0) slot = atomicAdd(b.ctrl + 4, n);
        slot = __shfl_sync(0xffffffffu, slot, 0);
        if (slot + n > b.capacity) n = 0;                          // cannot happen: capacity = pairs of the job
        if (lane == 0) { b.row_slot[2 * row] = slot; b.row_slot[2 * row + 1] = n; }
        if (n == 0) continue;
        uint32_t k = slot;
        for (uint32_t h0 = 0; h0 < rg.nhaps; h0 += 32) {
            const bool fail = h0 + lane < rg.nhaps && raw[h0 + lane] < b.threshold;
            const unsigned m = __ballot_sync(0xffffffffu, fail);
            if (fail) {
                const uint32_t pos = k + __popc(m & lt);
                b.out_index[pos] = base + h0 + lane;
                b.hap_list[pos] = rg.hap_first + h0 + lane;
            }
            k += __popc(m);
        }
        __syncwarp();                                              // hap_list of this row is read back below
        const RowCut rc = cut_row(b, read, n, run_cap);
        for (uint32_t t = lane; t < rc.ntask; t += 32) atomicAdd(b.ctrl + kCtrlHist + task_class(b, slot, n, rc.ntask, t, run_cap), 1u);
    }
}

__global__ void __launch_bounds__(256) fallback_tasks_kernel(const FallbackBuild b)
{
    const uint32_t total = b.ctrl[0];
    if (total == 0) return;
    __shared__ uint32_t first[kCostClasses];                       // position of each class's first task
    if (threadIdx.x < 32) {
        static_assert(kCostClasses == 64, "two classes per lane");
        const uint32_t c0 = b.ctrl[kCtrlHist + 2 * threadIdx.x], c1 = b.ctrl[kCtrlHist + 2 * threadIdx.x + 1];
        uint32_t incl = c0 + c1;
        #pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o); if ((int)threadIdx.x >= o) incl += v; }
        first[2 * threadIdx.x] = incl - c0 - c1; first[2 * threadIdx.x + 1] = incl - c1;
        if (blockIdx.x == 0 && threadIdx.x == 31) b.ctrl[3] = incl;   // number of tasks, read by the double kernel
    }
    __syncthreads();
    const uint32_t run_cap = fallback_run_cap(b, total);
    const uint32_t lane = threadIdx.x & 31, warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; row < b.num_rows; row += warps) {
        const uint32_t slot = b.row_slot[2 * row], n = b.row_slot[2 * row + 1];
        if (n == 0) continue;
        RegionDesc rg; uint32_t read, base;
        row_of(b, row, rg, read, base);
        const RowCut rc = cut_row(b, read, n, run_cap);
        for (uint32_t t = lane; t < rc.ntask; t += 32) {
            const uint32_t cls = task_class(b, slot, n, rc.ntask, t, run_cap);
            const uint32_t pos = first[cls] + atomicAdd(b.ctrl + kCtrlClassCursor + cls, 1u);
            const uint32_t k0 = (uint32_t)((uint64_t)n * t / rc.ntask), k1 = (uint32_t)((uint64_t)n * (t + 1) / rc.ntask);
            Task tk;
            tk.read[0] = read; tk.read[1] = tk.read[2] = tk.read[3] = 0;
            tk.out_base[0] = slot + k0; tk.out_base[1] = tk.out_base[2] = tk.out_base[3] = 0;
            tk.hap_first = slot + k0; tk.nhaps = k1 - k0; tk.nreads = 1; tk.param_off = 0;
            b.tasks[pos] = tk;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// Row parameters of the float pass: one CTA per read group, see GroupDesc in pmm_types.h for the layout.
// What the reference recomputes for every pair (initializeVectors, avx-pairhmm-template.h:108-127, and the
// 1 - distm, distm / 3 of stripeINITIALIZATION, :155-158) is done here once per read.
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) read_params_kernel(const uint8_t* __restrict__ blob, const ReadDesc* __restrict__ reads,
                                                          const GroupDesc* __restrict__ groups, uint32_t ngroups,
                                                          DeviceTables tab, float* __restrict__ params)
{
    if (blockIdx.x >= ngroups) return;
    // the quality -> probability table is looked up four times per row: staged in shared memory
    __shared__ float s_ph2pr[128];
    if (threadIdx.x < 128) s_ph2pr[threadIdx.x] = __ldg(tab.ph2pr_f + threadIdx.x);
    __syncthreads();
    const GroupDesc gd = groups[blockIdx.x];
    const uint32_t K = gd.K, W = gd.W, KW = K * W, rows = gd.nstripes * KW;
    const uint32_t slots = gd.nstripes > 1 ? 1u : 32u / W;
    for (uint32_t slot = 0; slot < slots; ++slot) {
        const bool valid = slot < gd.nreads;
        ReadDesc rd = {0u, 0u, 0u};
        if (valid) rd = reads[gd.read[slot]];
        const int pad = (int)rows - (int)rd.len;                 // boundary rows above the read (all rows if unused)
        float* base = params + gd.param_off + (size_t)slot * gd.nstripes * kParamPlanes * KW;
        for (uint32_t x = threadIdx.x; x < rows; x += blockDim.x) {
            const uint32_t s = x / KW, idx = x % KW, j = idx / W, l = idx % W;
            const int r0 = (int)(s * KW + l * K + j) - pad;      // 0-based read base of row j of lane l
            float v[kParamPlanes] = {0.f, 0.f, 0.f, 0.f, 1.0f, 0.f, 0.f, __uint_as_float(kPadClass)};
            if (valid && r0 >= 0) {
                const uint8_t* b = blob + rd.off + r0;
                const int q_ = b[rd.stride] & 127, i_ = b[2 * rd.stride] & 127;
                const int d_ = b[3 * rd.stride] & 127, c_ = b[4 * rd.stride] & 127;
                const int mx = max(i_, d_), mn = min(i_, d_);
                const float pc = s_ph2pr[c_], dm = s_ph2pr[q_];
                v[0] = __ldg(tab.m2m_f + ((mx * (mx + 1)) >> 1) + mn);
                v[1] = __fsub_rn(1.0f, pc);
                v[2] = s_ph2pr[i_];
                v[3] = s_ph2pr[d_];
                v[4] = pc;
                v[5] = __fsub_rn(1.0f, dm);
                v[6] = __fdiv_rn(dm, 3.0f);
                v[7] = __uint_as_float((unsigned)base_class(b[0]));
            }
            float* o = base + (size_t)s * kParamPlanes * KW + idx;
            #pragma unroll
            for (int p = 0; p < kParamPlanes; ++p) o[(size_t)p * KW] = v[p];
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// Haplotype stream builder: one CTA per haplotype.
// ---------------------------------------------------------------------------------------------------------
__global__ void build_stream_kernel(const uint8_t* __restrict__ blob, const HapDesc* __restrict__ haps,
                                    const uint32_t* __restrict__ spos, uint32_t num_hap, uint8_t* __restrict__ stream,
                                    float* __restrict__ iy_f, double* __restrict__ iy_d, float ic_f, double ic_d)
{
    const uint32_t h = blockIdx.x;
    if (h >= num_hap) return;
    const HapDesc d = haps[h];
    uint8_t* dst = stream + spos[h];
    if (threadIdx.x == 0) {
        dst[0] = kSep;
        // INITIAL_CONSTANT / haplen with the int converted to NUMBER first (avx-pairhmm-template.h:86)
        iy_f[h] = __fdiv_rn(ic_f, (float)(int)d.len);
        iy_d[h] = __ddiv_rn(ic_d, (double)(int)d.len);
        if (h + 1 == num_hap) dst[1 + d.len] = kSep;
    }
    for (uint32_t k = threadIdx.x; k < d.len; k += blockDim.x) dst[1 + k] = (uint8_t)base_class(blob[d.off + k]);
}

// ---------------------------------------------------------------------------------------------------------
// FP32 issue-rate probe (roofline denominator): 8 independent FMUL/FADD chains per thread.
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) fp32_probe_kernel(float* sink, int iters)
{
    float x[8];
    #pragma unroll
    for (int i = 0; i < 8; ++i) x[i] = 1.0f + threadIdx.x * 1e-3f + i;
    const float m = 0.99999f, c = 1e-6f;
    for (int it = 0; it < iters; ++it) {
        // 512 FP32 instructions per trip: the three loop instructions cost 0.6 % of the issue slots (with 64 per trip
        // the probe under-reported the peak by 4.5 %)
        #pragma unroll
        for (int rep = 0; rep < 64; ++rep) {
            #pragma unroll
            for (int i = 0; i < 8; ++i) x[i] = (rep & 1) ? __fadd_rn(x[i], c) : __fmul_rn(x[i], m);
        }
    }
    float s = 0;
    #pragma unroll
    for (int i = 0; i < 8; ++i) s += x[i];
    sink[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

// The same for the FP64 pipe (roofline denominator of the double re-run): independent DMUL/DADD chains.
__global__ void __launch_bounds__(256) fp64_probe_kernel(double* sink, int iters)
{
    double x[8];
    #pragma unroll
    for (int i = 0; i < 8; ++i) x[i] = 1.0 + threadIdx.x * 1e-3 + i;
    const double m = 0.99999, c = 1e-6;
    for (int it = 0; it < iters; ++it) {
        #pragma unroll
        for (int rep = 0; rep < 64; ++rep) {
            #pragma unroll
            for (int i = 0; i < 8; ++i) x[i] = (rep & 1) ? __dadd_rn(x[i], c) : __dmul_rn(x[i], m);
        }
    }
    double s = 0;
    #pragma unroll
    for (int i = 0; i < 8; ++i) s += x[i];
    sink[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

// ---------------------------------------------------------------------------------------------------------
// Variant table
// ---------------------------------------------------------------------------------------------------------
// The shared-memory attribute and the occupancy of a variant are per device and never change: looked up once per
// (variant, device) instead of on every launch (runtime calls that take the driver's locks, which feeder threads of
// eight GPUs in one process would otherwise contend for several times per job).
constexpr int kMaxDevices = 64;
inline int current_device() { int d = 0; if (cudaGetDevice(&d) != cudaSuccess || d < 0 || d >= kMaxDevices) d = -1; return d; }

// dynamic shared memory of a variant: the weight tables of its warps
template <typename T, int K> constexpr int variant_smem() { return kWarpsPerCta * wtab_elems<T, K>() * (int)sizeof(T); }

template <typename T, int K, int W, bool STRIPED, int F>
cudaError_t prepare_variant()
{
    static std::atomic<bool> ready[kMaxDevices];
    const int dev = current_device();
    if (dev >= 0 && ready[dev].load(std::memory_order_acquire)) return cudaSuccess;
    const cudaError_t e = cudaFuncSetAttribute(pmm_forward_kernel<T, K, W, STRIPED, F>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                               variant_smem<T, K>());
    if (e == cudaSuccess && dev >= 0) ready[dev].store(true, std::memory_order_release);
    return e;
}

template <typename T, int K, int W, bool STRIPED, int F>
cudaError_t launch_variant(const ForwardArgs& a, const FallbackQueue& fq, int ctas, cudaStream_t s)
{
    const cudaError_t e = prepare_variant<T, K, W, STRIPED, F>();
    if (e != cudaSuccess) return e;
    pmm_forward_kernel<T, K, W, STRIPED, F><<<ctas, kWarpsPerCta * 32, variant_smem<T, K>(), s>>>(a, fq);
    return cudaGetLastError();
}

template <typename T, int K, int W, bool STRIPED, int F>
int variant_ctas_per_sm()
{
    static std::atomic<int> cached[kMaxDevices];               // occupancy + 1; 0 = not looked up yet
    const int dev = current_device();
    if (dev >= 0) { const int v = cached[dev].load(std::memory_order_relaxed); if (v) return v - 1; }
    if (prepare_variant<T, K, W, STRIPED, F>() != cudaSuccess) return 0;
    int n = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, pmm_forward_kernel<T, K, W, STRIPED, F>, kWarpsPerCta * 32,
                                                      variant_smem<T, K>()) != cudaSuccess) return 0;
    if (dev >= 0) cached[dev].store(n + 1, std::memory_order_relaxed);
    return n;
}

template <typename T, int K, int W, bool STRIPED, int F>
constexpr ForwardKernel kVariant{&variant_ctas_per_sm<T, K, W, STRIPED, F>, &launch_variant<T, K, W, STRIPED, F>};

}  // namespace

const ForwardKernel* forward_f32_variant(int K, int W, bool striped, bool fast)
{
    if (striped) {
        if (K != kStripedK || W != 32) return nullptr;
        return fast ? &kVariant<float, kStripedK, 32, true, kPush | kFast> : &kVariant<float, kStripedK, 32, true, kPush>;
    }
#define X(k, w) if (K == k && W == w) return fast ? &kVariant<float, k, w, false, kPush | kFast> : &kVariant<float, k, w, false, kPush>;
    PMM_F32_VARIANTS(X)
#undef X
    return nullptr;
}

// Exact float re-check of single pairs (fast mode's guard band): one read per warp, any length, parameters inline.
const ForwardKernel& recheck_f32_variant() { return kVariant<float, kStripedK, 32, true, kPush | kInline>; }

// striped = false: every read of the job fits one stripe (32 K - 1 bases), the common case; the loop then carries no
// row through scratch memory (in the striped variant those loads, stores and their branches are a fifth of the
// steady loop's non-DP instructions).
const ForwardKernel* forward_f64_variant(int K, bool striped)
{
#define X(k) if (K == k) return striped ? &kVariant<double, k, 32, true, kRetry | kList> : &kVariant<double, k, 32, false, kRetry | kList>;
    PMM_F64_ROWS(X)
#undef X
    return nullptr;
}

// Rows per lane of the double kernel for a job whose longest read has max_read_len bases: the block (128, 160, 192 or
// 256 rows per stripe) that wastes the fewest rows on it; ties go to the larger block (fewer stripes, shorter chain).
int pick_f64_rows(uint32_t max_read_len)
{
    const uint32_t rows = max_read_len + 1;
    int best = 0; uint32_t best_padded = 0;
    for (int k : kF64Rows) {
        const uint32_t blk = 32u * k, padded = (rows + blk - 1) / blk * blk;
        if (!best || padded <= best_padded) { best = k; best_padded = padded; }
    }
    return best;
}

cudaError_t launch_build_fallback(const FallbackBuild& b, int sm_count, cudaStream_t s)
{
    if (b.num_rows == 0) return cudaSuccess;
    const int ctas = (int)std::min<uint64_t>(((uint64_t)b.num_rows + 7) / 8, (uint64_t)sm_count * 8);
    fallback_scan_kernel<<<ctas, 256, 0, s>>>(b);
    fallback_tasks_kernel<<<ctas, 256, 0, s>>>(b);
    return cudaGetLastError();
}

cudaError_t launch_build_stream(const uint8_t* hap_blob, const HapDesc* haps, const uint32_t* spos, uint32_t num_hap,
                                uint8_t* stream, float* inity_f, double* inity_d, float ic_f, double ic_d,
                                cudaStream_t s)
{
    if (num_hap == 0) return cudaSuccess;
    build_stream_kernel<<<num_hap, 128, 0, s>>>(hap_blob, haps, spos, num_hap, stream, inity_f, inity_d, ic_f, ic_d);
    return cudaGetLastError();
}

cudaError_t launch_read_params(const uint8_t* read_blob, const ReadDesc* reads, const GroupDesc* groups, uint32_t ngroups,
                               const DeviceTables& tab, float* params, cudaStream_t s)
{
    if (ngroups == 0) return cudaSuccess;
    read_params_kernel<<<ngroups, 128, 0, s>>>(read_blob, reads, groups, ngroups, tab, params);
    return cudaGetLastError();
}

cudaError_t launch_fp32_probe(float* sink, int iters, int ctas, cudaStream_t s)
{
    fp32_probe_kernel<<<ctas, 256, 0, s>>>(sink, iters);
    return cudaGetLastError();
}

cudaError_t launch_fp64_probe(double* sink, int iters, int ctas, cudaStream_t s)
{
    fp64_probe_kernel<<<ctas, 256, 0, s>>>(sink, iters);
    return cudaGetLastError();
}

}  // namespace pmm
