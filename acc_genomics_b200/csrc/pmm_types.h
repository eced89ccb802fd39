// pmm_types.h -- plain data shared by the host planner (pmm_plan.cpp), the engine and the kernels.  No CUDA here.
#pragma once
#include <cstdint>

namespace pmm {

constexpr int kMaxGroups = 4;           // reads per warp: 32 / W, W >= 8
// Warps per CTA of the forward kernels.  Every warp works alone (its own tasks, its own slice of shared memory; no
// __syncthreads anywhere), so the CTA size only decides the granularity at which the SM's registers and shared memory are
// taken and given back.  Measured with 1: no difference anywhere -- in particular a one-warp CTA of the double kernel does
// not slip in beside the float kernel's eight warps per SM, because registers are per SMSP (16 384 each, two float warps
// of 7 424 leave 1 536): DESIGN.md section 4.5.
constexpr int kWarpsPerCta = 4;
constexpr int kF64K = 6;                // rows per lane of the double kernel (W = 32): 191-base reads in one stripe
constexpr int kMaxK = 20;               // most rows per lane of any float variant
constexpr int kStripedK = 8;            // rows per lane of the striped float kernel (W = 32)
// Rows per lane of the double kernel's instantiations (W = 32), of which pick_f64_rows() chooses one per job.
#define PMM_F64_ROWS(X) X(4) X(5) X(6) X(8)
#define PMM_F64_ROWS_ITEM(k) k,
constexpr int kF64Rows[] = {PMM_F64_ROWS(PMM_F64_ROWS_ITEM)};
#undef PMM_F64_ROWS_ITEM

// Resident CTAs per SM of the forward kernel for element type T and K rows per lane: what its __launch_bounds__ asks the
// register allocator to leave room for, and what the planner counts on.  The state of a lane is 8 registers per row
// (5 parameters + M, X, Y), so K decides the occupancy step (64K registers / 128 threads).
// Measured (tools/occ_check.py): 15 and 16 rows per lane at two CTAs per SM (up to 255 registers) beat three CTAs at 168
// registers by 5.6 % (config 4, K = 16 / W = 16: 2 343 -> 2 475 GCUPS); for K <= 14 the difference is within 2 %.
template <typename T> constexpr int resident_ctas(int K)
{
    return sizeof(T) == 8 ? (K <= 6 ? 3 : 2) : K <= 11 ? 4 : K <= 14 ? 3 : 2;
}

struct ReadDesc { uint32_t off, stride, len; };
struct HapDesc  { uint32_t off, len; };
struct RegionDesc { uint32_t read_first, nreads, hap_first, nhaps, out_first, row_first; };   // row_first: reads of earlier regions

// One unit of work for one warp.  Group g (lanes g*W .. g*W+W-1) owns read[g]; all groups walk the same run of
// haplotypes [hap_first, hap_first + nhaps).  The result for (read[g], hap_first + n) goes to out[out_base[g] + n].
// List tasks (the double re-run): one read; hap_first indexes the fallback list, whose entries hap_first .. hap_first +
// nhaps - 1 name the haplotypes, and out_base[0] is the first of the task's slots (= hap_first).
struct Task {
    uint32_t read[kMaxGroups];
    uint32_t out_base[kMaxGroups];
    uint32_t hap_first;
    uint32_t nhaps;
    uint32_t nreads;
    uint32_t param_off;                 // float pass: index (in floats) of the group's row parameters, see GroupDesc
};
static_assert(sizeof(Task) == 48, "Task layout");

// Row parameters per read are computed once per job (not once per pair like the reference's initializeVectors,
// avx-pairhmm-template.h:83-128) by read_params_kernel and stored per read group in the order the forward kernel's
// lanes consume them.  A group is the set of up to 32/W reads that share a warp.  Slot g of the group owns
// nstripes * kParamPlanes * K * W floats starting at param_off + g * nstripes * kParamPlanes * K * W, laid out
// [stripe][plane][j][l]: plane p of the row that is row j of lane l -- consecutive lanes read consecutive addresses.
// Planes: 0 pMM, 1 pGAPM, 2 pMX, 3 pMY, 4 pXX = pYY, 5 match weight 1 - e, 6 mismatch weight e / 3, 7 base class
// as an integer (0..4, kPadClass for a boundary row above the read or an unused slot).
constexpr int kParamPlanes = 8;
constexpr uint32_t kPadClass = 5;
struct GroupDesc {
    uint32_t read[kMaxGroups];
    uint32_t nreads;
    uint32_t K, W, nstripes;            // nstripes > 1 only for the striped variant (one read per group)
    uint32_t param_off;
    uint32_t reserved[3];
};
static_assert(sizeof(GroupDesc) == 48, "GroupDesc layout");

// (K rows per lane, W lanes per read) instantiations of the float kernel.
#define PMM_F32_VARIANTS(X) \
    X(4, 8) X(5, 8) X(6, 8) X(7, 8) X(8, 8) X(9, 8) X(10, 8) X(11, 8) X(12, 8) X(13, 8) X(14, 8) X(15, 8) X(16, 8) \
    X(17, 8) X(18, 8) X(19, 8) X(20, 8) \
    X(4, 16) X(5, 16) X(6, 16) X(7, 16) X(8, 16) X(9, 16) X(10, 16) X(11, 16) X(12, 16) X(14, 16) X(16, 16) \
    X(4, 32) X(5, 32) X(6, 32) X(7, 32) X(8, 32) X(9, 32) X(10, 32) X(12, 32) X(14, 32) X(16, 32)

inline bool forward_f32_has_variant(int K, int W)
{
#define PMM_X(k, w) if (K == k && W == w) return true;
    PMM_F32_VARIANTS(PMM_X)
#undef PMM_X
    return false;
}

struct Variant { int K, W; bool striped; };
inline bool operator==(const Variant& a, const Variant& b) { return a.K == b.K && a.W == b.W && a.striped == b.striped; }

}  // namespace pmm
