// pmm_engine.cu -- the C ABI of include/pairhmm_cuda.h: host-side packing, task queue construction, kernel
// sequencing, result collection.  This is the layer that stands where the reference has pack_fpga_input +
// OpenCL buffer migration + clEnqueueTask (/root/reference/pairhmm/task/xlnx/PairHMMTask.cpp:27-143,
// /root/reference/pairhmm/host/PairHMMFpga.cpp:125-162).  There is no CPU compute path in this file: without a
// GPU every entry point fails with PMM_ERR_NO_DEVICE.
#include "../../include/pairhmm_cuda.h"
#include "cuda_util.h"
#include "host_workers.h"
#include "pmm_kernels.cuh"
#include "pmm_plan.h"
#include "pmm_tables.h"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

using namespace pmm;

namespace {

thread_local std::string g_create_error;      // last error of the calls that have no context (pmm_create, pmm_plan_flat), per thread

constexpr size_t kAlign = 256;
constexpr uint32_t kCtrlWords = kCtrlCursors + 32 * 104;
inline size_t align_up(size_t x) { return (x + kAlign - 1) / kAlign * kAlign; }

// Typed pointer to the section at byte offset `off` of a buffer (host or device side of the input arena).
template <class T> T* section(void* base, size_t off) { return reinterpret_cast<T*>(static_cast<char*>(base) + off); }

// The input arena, one H2D copy per job: read blob | descs | hap blob | descs | spos | tasks | regions | groups.
struct ArenaLayout { size_t rblob = 0, rdesc = 0, hblob = 0, hdesc = 0, spos = 0, tasks = 0, regions = 0, groups = 0, bytes = 0; };
ArenaLayout arena_layout(size_t rblob_bytes, uint32_t num_read, size_t hblob_bytes, uint32_t num_hap, uint64_t num_tasks,
                         uint32_t num_region, size_t num_groups)
{
    ArenaLayout a;
    size_t off = 0;
    auto put = [&](size_t& at, size_t bytes) { at = off; off = align_up(off + bytes); };
    put(a.rblob, rblob_bytes);
    put(a.rdesc, sizeof(ReadDesc) * num_read);
    put(a.hblob, hblob_bytes);
    put(a.hdesc, sizeof(HapDesc) * num_hap);
    put(a.spos, sizeof(uint32_t) * (num_hap + 1));
    put(a.tasks, sizeof(Task) * num_tasks);
    put(a.regions, sizeof(RegionDesc) * num_region);
    put(a.groups, sizeof(GroupDesc) * num_groups);
    a.bytes = off;
    return a;
}

// The pinned block a launch's results are copied to: 256-byte header (control words) | raw floats | fallback indices |
// doubles of the fallback pairs.
struct OutLayout { size_t raw, idx, dres, bytes; };
OutLayout out_layout(uint64_t pairs)
{
    OutLayout o;
    o.raw = 256;
    o.idx = o.raw + align_up(sizeof(float) * pairs);
    o.dres = o.idx + align_up(sizeof(uint32_t) * pairs);
    o.bytes = o.dres + sizeof(double) * pairs + 256;
    return o;
}

// What pmm_stage_* leaves for pmm_launch and the fetches; every stage replaces it as a whole.
struct StagedJob {
    ArenaLayout at;                     // sections of the input arena
    uint32_t num_region = 0, num_groups = 0, num_tasks = 0, num_rows = 0;
    uint64_t pairs = 0;
    uint32_t max_hap_len = 0;
    std::vector<LaunchSeg> segs;        // one float-kernel launch each
    int f64_rows = kF64K;               // rows per lane of the double kernel (pick_f64_rows) ...
    bool f64_striped = true;            // ... and whether its longest read needs more than one stripe of 32 x rows
};

// A job as stage() takes it.  read_off / hap_off (num + 1 entries) and the regions are what the planner reads; the
// device-side blobs are the concatenation of read_parts / hap_parts, and the descriptors give every read's five tracks
// (off, stride, len) and every haplotype (off, len) inside those blobs.  The context keeps one, reused by every job: the
// flat builder points read_off, hap_off and regions at the caller's arrays, the other builders at roff, hoff and
// own_regions.
struct BlobPart { const uint8_t* p; size_t n; };
struct JobSource {
    uint32_t num_read = 0, num_hap = 0, num_region = 0;
    const uint32_t* read_off = nullptr;
    const uint32_t* hap_off = nullptr;
    const pmm_region_t* regions = nullptr;
    std::vector<BlobPart> read_parts, hap_parts;
    std::vector<ReadDesc> rdesc;
    std::vector<HapDesc> hdesc;
    std::vector<uint32_t> roff, hoff;
    std::vector<pmm_region_t> own_regions;

    void reset()
    {
        roff.assign(1, 0); hoff.assign(1, 0);
        rdesc.clear(); hdesc.clear(); read_parts.clear(); hap_parts.clear(); own_regions.clear();
    }
    // Reads and haplotypes gathered from the caller's pointers: the five tracks of a read back to back, like the wire
    // format.
    void add_read(const char* const tracks[5], uint32_t len)
    {
        rdesc.push_back(ReadDesc{(uint32_t)(5ull * roff.back()), len, len});
        roff.push_back(roff.back() + len);
        for (int t = 0; t < 5; ++t) read_parts.push_back(BlobPart{reinterpret_cast<const uint8_t*>(tracks[t]), len});
    }
    void add_hap(const char* bases, uint32_t len)
    {
        hdesc.push_back(HapDesc{hoff.back(), len});
        hoff.push_back(hoff.back() + len);
        hap_parts.push_back(BlobPart{reinterpret_cast<const uint8_t*>(bases), len});
    }
    void use_own_arrays()
    {
        num_read = (uint32_t)rdesc.size(); num_hap = (uint32_t)hdesc.size(); num_region = (uint32_t)own_regions.size();
        read_off = roff.data(); hap_off = hoff.data(); regions = own_regions.data();
    }
};

}  // namespace

// What one launch produces, twice per context: launch i + 1's float pass runs while launch i's double re-run is still on
// the GPU (on its own stream), so the two must not share results, fallback lists, control words or the pinned block the
// results are copied to.  A fetch always refers to the set of the last launch.
struct ResultSet {
    DevBuf d_raw, d_fb_tasks, d_fb_idx, d_fb_hap, d_fb_rows, d_dres, d_ctrl;
    PinBuf h_out;                       // see out_layout
    cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};    // launch starts, float pass over, double re-run over
    cudaEvent_t ev_raw = nullptr, ev_lists = nullptr;   // the copies out of this set are over (its next user waits for them)
};

namespace {
struct HostOut { uint32_t* ctrl; float* raw; uint32_t* idx; double* dres; };
HostOut host_out(const ResultSet& r, uint64_t pairs)
{
    const OutLayout l = out_layout(pairs);
    return HostOut{section<uint32_t>(r.h_out.p, 0), section<float>(r.h_out.p, l.raw), section<uint32_t>(r.h_out.p, l.idx),
                   section<double>(r.h_out.p, l.dres)};
}
}  // namespace

struct pmm_ctx {
    int device = 0;
    int sm_count = 0;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    cudaStream_t f64_stream = nullptr;  // fallback builders + double re-run: next to the following launch's float pass
    cudaStream_t copy_stream = nullptr; // D2H of the raw floats as soon as the float pass is over, under the double pass
    cudaStream_t list_stream = nullptr; // D2H of the control words and the fallback list behind the double pass
    ResultSet rs[2];
    int cur = 0;                        // set of the last launch
    ResultSet& R() { return rs[cur]; }
    const ResultSet& R() const { return rs[cur]; }
    cudaEvent_t ev_h2d = nullptr;       // recorded after the input arena's H2D copy; the next stage waits before repacking
    bool h2d_pending = false;
    cudaEvent_t ev_ref = nullptr;       // recorded and waited for in pmm_create: origin of the context's device timeline ...
    double ref_host_s = 0;              // ... and the host's steady clock at that moment (pmm_get_timeline)
    cudaEvent_t ev_probe = nullptr;     // issue-rate probes
    cudaEvent_t ev_block = nullptr;     // "sync" = "block": waits sleep on this event instead of spinning on the stream
    cudaEvent_t ev_poll = nullptr;      // "sync" = "auto": spun on or polled
    bool block_sync = false;
    int spin_us = 0;                    // "sync" = "hybrid": poll this long, then sleep on the blocking event
    bool auto_sync = false;             // "sync" = "auto": spin while few threads of the process do, else sleep
    std::string err;
    PlanOptions plan_opt = plan_defaults();   // how stage() cuts jobs into warp-tasks (pmm_set_option)
    bool fast = false;                  // "mode" option: fast = contracted float kernels + exact re-check near the threshold
    float guard = 0.0078125f;           // "guard" option: relative half-width of the re-check band around 1e-28f (2^-7)
    int f64_tasks_per_warp = 6;         // "f64_tasks_per_warp": tasks the double re-run aims at per resident warp ...
    int f64_max_run = 6;                // "f64_max_run": ... and the most haplotypes it puts into one task (tools/f64_sweep.py)
    bool overlap = true;                // "overlap": consecutive launches overlap by one pass (off: a launch ends with its own re-run)

    // device-resident tables
    DevBuf tables;
    DeviceTables dtab{};

    // job state
    PinBuf h_in;  DevBuf d_in;          // the input arena, see arena_layout
    DevBuf d_params, d_stream, d_iyf, d_iyd, d_tiny_tasks, d_scratch, d_scratch64, d_probe;
    StagedJob job;
    bool staged = false, launched = false;
    bool have_raw = false, have_lists = false;   // what of the last launch's results is already in h_out
    uint32_t spec = 0;                           // fallback entries copied back speculatively by pmm_launch
    pmm_stats_t stats{};
    JobSource src;                               // scratch of the job builders, reused from job to job

    int fail_cuda(cudaError_t e, const char* what)
    {
        err = std::string(what) + ": " + cudaGetErrorString(e);
        return PMM_ERR_CUDA;
    }
    int fail(int code, const std::string& m) { err = m; return code; }
};

#define PMM_CUDA(ctx, call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return (ctx)->fail_cuda(e__, #call); } while (0)

namespace {

int ensure_tables(pmm_ctx* c)
{
    if (c->tables.p) return PMM_OK;
    const HostTables& t = host_tables();
    const size_t nf = kPh2prSize + kM2mSize;
    const size_t bytes = align_up(nf * sizeof(float)) + nf * sizeof(double);
    PMM_CUDA(c, c->tables.reserve(bytes));
    char* base = static_cast<char*>(c->tables.p);
    float* f = reinterpret_cast<float*>(base);
    double* d = reinterpret_cast<double*>(base + align_up(nf * sizeof(float)));
    PMM_CUDA(c, cudaMemcpy(f, t.ph2pr_f, sizeof t.ph2pr_f, cudaMemcpyHostToDevice));
    PMM_CUDA(c, cudaMemcpy(f + kPh2prSize, t.m2m_f, sizeof t.m2m_f, cudaMemcpyHostToDevice));
    PMM_CUDA(c, cudaMemcpy(d, t.ph2pr_d, sizeof t.ph2pr_d, cudaMemcpyHostToDevice));
    PMM_CUDA(c, cudaMemcpy(d + kPh2prSize, t.m2m_d, sizeof t.m2m_d, cudaMemcpyHostToDevice));
    c->dtab = DeviceTables{f, f + kPh2prSize, d, d + kPh2prSize};
    return PMM_OK;
}

// The one staging path: plan the job, lay out and fill the pinned input arena, reserve the device buffers, enqueue the
// H2D copy and the haplotype stream build.
int stage(pmm_ctx* c, const JobSource& src)
{
    auto t0 = std::chrono::steady_clock::now();
    cudaSetDevice(c->device);
    c->staged = false; c->launched = false;
    // the pinned input arena is about to be repacked: the previous job's H2D copy out of it must be over
    // (stage, launch, stage with no fetch in between)
    if (c->h2d_pending) { PMM_CUDA(c, cudaEventSynchronize(c->ev_h2d)); c->h2d_pending = false; }
    // ... and the device-side inputs are about to be overwritten: the double re-runs of earlier launches read them on
    // their own stream
    for (ResultSet& r : c->rs) PMM_CUDA(c, cudaStreamWaitEvent(c->stream, r.ev[2], 0));
    int rc = ensure_tables(c);
    if (rc) return rc;

    size_t sz_rblob = 0, sz_hblob = 0;
    for (const BlobPart& bp : src.read_parts) sz_rblob += bp.n;
    for (const BlobPart& bp : src.hap_parts) sz_hblob += bp.n;
    StagedJob job;
    cudaError_t arena_err = cudaSuccess;

    // The planner calls back once it knows how many tasks and groups there are; the input arena is laid out and
    // reserved then, and the tasks are written straight into pinned memory (no intermediate copy).
    Plan plan;
    {
        std::string perr;
        rc = plan_job(src.num_read, src.read_off, src.num_hap, src.hap_off, src.num_region, src.regions, c->sm_count, c->plan_opt,
                      plan, perr, [&](const Plan& p) -> Task* {
            job.at = arena_layout(sz_rblob, src.num_read, sz_hblob, src.num_hap, p.num_tasks, src.num_region, p.groups.size());
            if ((arena_err = c->h_in.reserve(job.at.bytes)) != cudaSuccess) return nullptr;
            if ((arena_err = c->d_in.reserve(job.at.bytes)) != cudaSuccess) return nullptr;
            return section<Task>(c->h_in.p, job.at.tasks);
        });
        if (arena_err != cudaSuccess) return c->fail_cuda(arena_err, "input arena");
        if (rc) return c->fail(rc, perr);
    }
    static const bool trace = getenv("PMM_TRACE_STAGE") != nullptr;       // phase times of staging on stderr
    const auto t_plan = std::chrono::steady_clock::now();
    const ArenaLayout& at = job.at;
    const uint64_t pairs = plan.pairs;
    job.num_region = src.num_region; job.num_groups = (uint32_t)plan.groups.size();
    job.num_tasks = (uint32_t)plan.num_tasks; job.num_rows = (uint32_t)plan.rows;
    job.pairs = pairs;
    job.max_hap_len = plan.max_hap_len;
    job.segs = std::move(plan.segs);
    job.f64_rows = pick_f64_rows(plan.max_read_len);
    job.f64_striped = plan.max_read_len + 1 > 32u * (uint32_t)job.f64_rows;

    // ---- pack the rest of the input arena ---------------------------------------------------------------------
    {
        uint8_t* w = section<uint8_t>(c->h_in.p, at.rblob);
        for (const BlobPart& bp : src.read_parts) { memcpy(w, bp.p, bp.n); w += bp.n; }
        w = section<uint8_t>(c->h_in.p, at.hblob);
        for (const BlobPart& bp : src.hap_parts) { memcpy(w, bp.p, bp.n); w += bp.n; }
    }
    memcpy(section<ReadDesc>(c->h_in.p, at.rdesc), src.rdesc.data(), sizeof(ReadDesc) * src.num_read);
    memcpy(section<HapDesc>(c->h_in.p, at.hdesc), src.hdesc.data(), sizeof(HapDesc) * src.num_hap);
    uint32_t* spos = section<uint32_t>(c->h_in.p, at.spos);
    uint32_t pos = 0;
    for (uint32_t h = 0; h < src.num_hap; ++h) { spos[h] = pos; pos += src.hdesc[h].len + 1; }
    spos[src.num_hap] = pos;                       // final separator
    memcpy(section<RegionDesc>(c->h_in.p, at.regions), plan.regions.data(), sizeof(RegionDesc) * src.num_region);
    memcpy(section<GroupDesc>(c->h_in.p, at.groups), plan.groups.data(), sizeof(GroupDesc) * plan.groups.size());

    const auto t_pack = std::chrono::steady_clock::now();
    // ---- device buffers -------------------------------------------------------------------------------------
    const size_t stream_bytes = kStreamFrontPad + (size_t)pos + 1 + kStreamTailPad;
    PMM_CUDA(c, c->d_stream.reserve(stream_bytes));
    PMM_CUDA(c, c->d_params.reserve(sizeof(float) * plan.param_floats));
    PMM_CUDA(c, c->d_iyf.reserve(sizeof(float) * src.num_hap));
    PMM_CUDA(c, c->d_iyd.reserve(sizeof(double) * src.num_hap));
    if (c->fast) PMM_CUDA(c, c->d_tiny_tasks.reserve(sizeof(Task) * pairs));     // re-check list of the guard band
    for (ResultSet& r : c->rs) {
        PMM_CUDA(c, r.d_raw.reserve(sizeof(float) * pairs));
        PMM_CUDA(c, r.d_fb_tasks.reserve(sizeof(Task) * pairs));
        PMM_CUDA(c, r.d_fb_idx.reserve(sizeof(uint32_t) * pairs));
        PMM_CUDA(c, r.d_fb_hap.reserve(sizeof(uint32_t) * pairs));
        PMM_CUDA(c, r.d_fb_rows.reserve(sizeof(uint32_t) * 2 * plan.rows));
        PMM_CUDA(c, r.d_dres.reserve(sizeof(double) * pairs));
        PMM_CUDA(c, r.d_ctrl.reserve(sizeof(uint32_t) * kCtrlWords));
        PMM_CUDA(c, r.h_out.reserve(out_layout(pairs).bytes));
    }
    // carry rows of the striped kernels: one haplotype (+2 separators) per warp, three rows of doubles
    {
        int ctas64 = 1;
        for (int k : kF64Rows) ctas64 = std::max(ctas64, forward_f64_variant(k, true)->ctas_per_sm());
        const int ctas32 = std::max({forward_f32_variant(kStripedK, 32, true, false)->ctas_per_sm(),
                                     forward_f32_variant(kStripedK, 32, true, true)->ctas_per_sm(), recheck_f32_variant().ctas_per_sm()});
        // the float and the double kernel of neighbouring launches can be on the GPU together: a scratch of their own each
        PMM_CUDA(c, c->d_scratch.reserve((size_t)c->sm_count * ctas32 * kWarpsPerCta * 3 * (size_t)(job.max_hap_len + 8) * sizeof(float)));
        PMM_CUDA(c, c->d_scratch64.reserve((size_t)c->sm_count * ctas64 * kWarpsPerCta * 3 * (size_t)(job.max_hap_len + 8) * sizeof(double)));
    }

    cudaStream_t s = c->stream;
    PMM_CUDA(c, cudaMemcpyAsync(c->d_in.p, c->h_in.p, at.bytes, cudaMemcpyHostToDevice, s));
    PMM_CUDA(c, cudaEventRecord(c->ev_h2d, s));
    c->h2d_pending = true;
    PMM_CUDA(c, cudaMemsetAsync(c->d_stream.p, 0, kStreamFrontPad, s));
    PMM_CUDA(c, cudaMemsetAsync(static_cast<char*>(c->d_stream.p) + kStreamFrontPad + pos + 1, 0, kStreamTailPad, s));
    const HostTables& ht = host_tables();
    PMM_CUDA(c, launch_build_stream(section<uint8_t>(c->d_in.p, at.hblob), section<HapDesc>(c->d_in.p, at.hdesc),
                                    section<uint32_t>(c->d_in.p, at.spos), src.num_hap,
                                    static_cast<uint8_t*>(c->d_stream.p) + kStreamFrontPad,
                                    static_cast<float*>(c->d_iyf.p), static_cast<double*>(c->d_iyd.p), ht.ic_f, ht.ic_d, s));

    c->stats = pmm_stats_t{};
    c->stats.pairs = pairs; c->stats.cells = plan.cells; c->stats.h2d_bytes = at.bytes; c->stats.f32_tasks = job.num_tasks;
    c->stats.ms_stage = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (trace) {
        auto us = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) { return std::chrono::duration<double, std::micro>(b - a).count(); };
        fprintf(stderr, "[stage] %u reads x %u haps, %zu tasks: plan %.0f us, pack %.0f us, reserve + enqueue %.0f us\n", src.num_read, src.num_hap,
                (size_t)plan.num_tasks, us(t0, t_plan), us(t_plan, t_pack), us(t_pack, std::chrono::steady_clock::now()));
    }
    c->job = std::move(job);
    c->staged = true;
    return PMM_OK;
}

// Walk one block of the reference's wire format (PairHMMHostInterface.cpp:175-207): a count, then per element a length
// word and `tracks` arrays of that many bytes (reads 5, haplotypes 1).  Calls each(offset of the first array, length).
template <class F> bool scan_wire(const uint8_t* p, uint64_t n, uint32_t tracks, F&& each)
{
    if (!p || n < 4) return false;
    int32_t num; memcpy(&num, p, 4);
    if (num < 0) return false;
    uint64_t pos = 4;
    if ((uint64_t)num > (n - 4) / 4) return false;          // every element takes at least its length word
    for (int32_t i = 0; i < num; ++i) {
        if (pos + 4 > n) return false;
        int32_t l; memcpy(&l, p + pos, 4); pos += 4;
        if (l < 0 || pos + (uint64_t)tracks * l > n) return false;
        each((uint32_t)pos, (uint32_t)l); pos += (uint64_t)tracks * l;
    }
    return true;
}

// ---- job builders: each fills c->src ------------------------------------------------------------------------

// Five flat tracks + one haplotype array, (offset, length) per element; the offsets and regions are the caller's.
void source_from_flat(JobSource& s, uint32_t num_read, const uint32_t* read_off, const uint8_t* const tracks[5],
                      uint32_t num_hap, const uint32_t* hap_off, const uint8_t* hap_bases, uint32_t num_region, const pmm_region_t* regions)
{
    const uint32_t r_base = read_off[0], h_base = hap_off[0];
    const size_t total_bases = read_off[num_read] - r_base, total_hap = hap_off[num_hap] - h_base;
    s.rdesc.resize(num_read); s.hdesc.resize(num_hap);
    for (uint32_t i = 0; i < num_read; ++i)
        s.rdesc[i] = ReadDesc{read_off[i] - r_base, (uint32_t)total_bases, read_off[i + 1] - read_off[i]};
    for (uint32_t h = 0; h < num_hap; ++h) s.hdesc[h] = HapDesc{hap_off[h] - h_base, hap_off[h + 1] - hap_off[h]};
    s.read_parts.clear();
    for (int t = 0; t < 5; ++t) s.read_parts.push_back(BlobPart{tracks[t] + r_base, total_bases});
    s.hap_parts.assign(1, BlobPart{hap_bases + h_base, total_hap});
    s.num_read = num_read; s.read_off = read_off;
    s.num_hap = num_hap; s.hap_off = hap_off;
    s.num_region = num_region; s.regions = regions;
}

// The wire format, one region: the blobs are the serialized buffers themselves (stride = len), which makes staging a
// serialized block one memcpy.
int source_from_serialized(pmm_ctx* c, const void* reads_ser, uint64_t reads_bytes, const void* haps_ser, uint64_t haps_bytes,
                           int* num_read, int* num_hap)
{
    JobSource& s = c->src;
    s.reset();
    const uint8_t* rp = static_cast<const uint8_t*>(reads_ser);
    const uint8_t* hp = static_cast<const uint8_t*>(haps_ser);
    const bool ok = scan_wire(rp, reads_bytes, 5, [&](uint32_t off, uint32_t len) {
                        s.rdesc.push_back(ReadDesc{off, len, len}); s.roff.push_back(s.roff.back() + len); }) &&
                    scan_wire(hp, haps_bytes, 1, [&](uint32_t off, uint32_t len) {
                        s.hdesc.push_back(HapDesc{off, len}); s.hoff.push_back(s.hoff.back() + len); });
    if (!ok) return c->fail(PMM_ERR_INVALID, "malformed serialized block");
    if (reads_bytes >= (1ull << 31) || haps_bytes >= (1ull << 31)) return c->fail(PMM_ERR_INVALID, "serialized block larger than 2 GiB");
    s.read_parts.assign(1, BlobPart{rp, (size_t)reads_bytes});
    s.hap_parts.assign(1, BlobPart{hp, (size_t)haps_bytes});
    const uint32_t nr = (uint32_t)s.rdesc.size(), nh = (uint32_t)s.hdesc.size();
    if (num_read) *num_read = (int)nr;
    if (num_hap) *num_hap = (int)nh;
    if (nr == 0 || nh == 0) return c->fail(PMM_ERR_INVALID, "empty batch");
    s.own_regions.assign(1, pmm_region_t{0, nr, 0, nh});
    s.use_own_arrays();
    return PMM_OK;
}

// pmm_read_t / pmm_hap_t arrays, one region: every track of every read is one part of the blob.
int source_from_structs(pmm_ctx* c, const pmm_read_t* reads, int num_read, const pmm_hap_t* haps, int num_hap)
{
    JobSource& s = c->src;
    s.reset();
    s.read_parts.reserve(5 * (size_t)num_read); s.hap_parts.reserve(num_hap);
    for (int i = 0; i < num_read; ++i) {
        const pmm_read_t& r = reads[i];
        if (r.len <= 0 || !r._b || !r._q || !r._i || !r._d || !r._c) return c->fail(PMM_ERR_INVALID, "read of length 0 or null track");
        const char* tr[5] = {r._b, r._q, r._i, r._d, r._c};
        s.add_read(tr, (uint32_t)r.len);
        if (5ull * s.roff.back() >= (1ull << 31)) return c->fail(PMM_ERR_INVALID, "batch larger than 2 GiB: split it");
    }
    for (int i = 0; i < num_hap; ++i) {
        if (haps[i].len <= 0 || !haps[i]._b) return c->fail(PMM_ERR_INVALID, "haplotype of length 0 or null");
        s.add_hap(haps[i]._b, (uint32_t)haps[i].len);
    }
    s.own_regions.assign(1, pmm_region_t{0, (uint32_t)num_read, 0, (uint32_t)num_hap});
    s.use_own_arrays();
    return PMM_OK;
}

// A GKL-shaped batch: one testcase per pair, pointers shared between the pairs of a read and of a haplotype.  Consecutive
// testcases with the same read are a row; consecutive rows with the same haplotype sequence are a region.  The results
// of the regions, read-major, are then exactly the testcases' order.
int source_from_testcases(pmm_ctx* c, const pmm_testcase_t* tc, uint64_t n)
{
    auto same_read = [](const pmm_testcase_t& a, const pmm_testcase_t& b) {
        return a.rs == b.rs && a.rslen == b.rslen && a.q == b.q && a.i == b.i && a.d == b.d && a.c == b.c; };
    JobSource& s = c->src;
    s.reset();
    uint64_t k = 0, prev_row = 0, prev_len = 0;        // previous row: testcases [prev_row, prev_row + prev_len)
    uint64_t hbytes = 0;
    bool have_prev = false;
    while (k < n) {
        uint64_t e = k + 1;
        while (e < n && same_read(tc[k], tc[e])) ++e;
        const pmm_testcase_t& t = tc[k];
        if (t.rslen <= 0 || !t.rs || !t.q || !t.i || !t.d || !t.c) return c->fail(PMM_ERR_INVALID, "read of length 0 or null track");
        bool same_haps = have_prev && e - k == prev_len;
        for (uint64_t z = 0; same_haps && z < e - k; ++z)
            same_haps = tc[k + z].hap == tc[prev_row + z].hap && tc[k + z].haplen == tc[prev_row + z].haplen;
        if (!same_haps) {
            // a new region: its haplotypes are this row's
            s.own_regions.push_back(pmm_region_t{(uint32_t)s.rdesc.size(), 0, (uint32_t)s.hdesc.size(), (uint32_t)(e - k)});
            for (uint64_t z = k; z < e; ++z) {
                if (tc[z].haplen <= 0 || !tc[z].hap) return c->fail(PMM_ERR_INVALID, "haplotype of length 0 or null");
                s.add_hap(tc[z].hap, (uint32_t)tc[z].haplen);
                hbytes += (uint32_t)tc[z].haplen;
            }
        }
        const char* tr[5] = {t.rs, t.q, t.i, t.d, t.c};
        s.add_read(tr, (uint32_t)t.rslen);
        if (5ull * s.roff.back() + hbytes >= (1ull << 31)) return c->fail(PMM_ERR_INVALID, "batch larger than 2 GiB: split it");
        s.own_regions.back().num_read++;
        prev_row = k; prev_len = e - k; have_prev = true;
        k = e;
    }
    uint64_t pairs = 0;
    for (const pmm_region_t& r : s.own_regions) pairs += (uint64_t)r.num_read * r.num_hap;
    if (pairs != n) return c->fail(PMM_ERR_INVALID, "internal: testcase grouping lost pairs");
    s.use_own_arrays();
    return PMM_OK;
}

}  // namespace

// The double re-run's stream, at the priority of the float pass's.  (Tried: one level above it, so that a re-run's blocks
// take freed slots before the next float pass's -- no difference in throughput on configs 2, 3 and 4 or through the pool,
// an FP32-pipe and an FP64-pipe kernel do not co-run to any advantage: the float pass leaves too few issue slots.)
static cudaError_t create_f64_stream(cudaStream_t* out, int prio)
{
    return cudaStreamCreateWithPriority(out, cudaStreamNonBlocking, prio);
}

// No exception crosses the C boundary (include/pairhmm_cuda.h): allocation failures of the host-side vectors and
// anything else thrown below an entry point become a status code and a message.
template <class F> static int guarded(pmm_ctx* c, F&& f)
{
    try { return f(); }
    catch (const std::bad_alloc&) {
        if (c) return c->fail(PMM_ERR_INVALID, "out of host memory");
        g_create_error = "out of host memory"; return PMM_ERR_INVALID;
    }
    catch (const std::exception& e) {
        if (c) return c->fail(PMM_ERR_INVALID, e.what());
        g_create_error = e.what(); return PMM_ERR_INVALID;
    }
}

// The one-shot entries: the job a builder left in c->src (`built` is the builder's status), staged, launched, fetched.
template <class Fetch> static int stage_launch_fetch(pmm_ctx* c, int built, Fetch&& fetch)
{
    int rc = built;
    if (rc || (rc = stage(c, c->src)) || (rc = pmm_launch(c))) return rc;
    return fetch();
}

// The peak probes: one warm-up launch(warm_iters), then the best of three timed launch(iters) of `ops` lane instructions
// each, in lane instructions per second.
template <class Launch> static int probe_rate(pmm_ctx* c, Launch&& launch, int warm_iters, int iters, double ops, double* rate)
{
    PMM_CUDA(c, launch(warm_iters));
    cudaEvent_t end;
    PMM_CUDA(c, cudaEventCreate(&end));
    double best = 0;
    cudaError_t e = cudaSuccess;
    for (int rep = 0; rep < 3 && e == cudaSuccess; ++rep) {
        e = cudaEventRecord(c->ev_probe, c->stream);
        if (e == cudaSuccess) e = launch(iters);
        if (e == cudaSuccess) e = cudaEventRecord(end, c->stream);
        if (e == cudaSuccess) e = cudaEventSynchronize(end);
        float ms = 0;
        if (e == cudaSuccess) { cudaEventElapsedTime(&ms, c->ev_probe, end); best = std::max(best, ops / (ms * 1e-3)); }
    }
    cudaEventDestroy(end);
    if (e != cudaSuccess) return c->fail_cuda(e, "peak probe");
    *rate = best;
    return PMM_OK;
}

// =========================================================================================================
extern "C" {

int pmm_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int pmm_create(int device, pmm_ctx** out)
{
    if (!out) return PMM_ERR_INVALID;
    *out = nullptr;
    int sm_count = 0;
    const int rc = open_device<PMM_ERR_INVALID, PMM_ERR_CUDA, PMM_ERR_NO_DEVICE>(device, sm_count, g_create_error, "this engine");
    if (rc) return rc;
    pmm_ctx* c = new pmm_ctx();
    c->device = device; c->sm_count = sm_count;
    cudaError_t e;
    if ((e = cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking)) != cudaSuccess) {
        g_create_error = cudaGetErrorString(e); delete c; return PMM_ERR_CUDA;
    }
    c->stream = c->own_stream;
    if ((e = cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking)) != cudaSuccess ||
        (e = cudaStreamCreateWithFlags(&c->list_stream, cudaStreamNonBlocking)) != cudaSuccess ||
        (e = create_f64_stream(&c->f64_stream, 0)) != cudaSuccess) {       // 0 = the default priority, like own_stream
        g_create_error = cudaGetErrorString(e);
        if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
        if (c->list_stream) cudaStreamDestroy(c->list_stream);
        cudaStreamDestroy(c->own_stream); delete c; return PMM_ERR_CUDA;
    }
    for (ResultSet& r : c->rs) {
        for (auto& ev : r.ev) cudaEventCreate(&ev);
        cudaEventCreateWithFlags(&r.ev_raw, cudaEventDisableTiming);
        cudaEventCreateWithFlags(&r.ev_lists, cudaEventDisableTiming);
    }
    cudaEventCreate(&c->ev_probe);
    cudaEventCreateWithFlags(&c->ev_block, cudaEventBlockingSync | cudaEventDisableTiming);
    cudaEventCreateWithFlags(&c->ev_poll, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&c->ev_h2d, cudaEventDisableTiming);
    cudaEventCreate(&c->ev_ref);
    cudaEventRecord(c->ev_ref, c->own_stream);
    cudaEventSynchronize(c->ev_ref);
    c->ref_host_s = std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
    *out = c;
    return PMM_OK;
}

void pmm_destroy(pmm_ctx* c)
{
    if (!c) return;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    if (c->f64_stream) cudaStreamSynchronize(c->f64_stream);
    if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
    if (c->list_stream) cudaStreamSynchronize(c->list_stream);
    for (ResultSet& r : c->rs) {
        for (auto& ev : r.ev) if (ev) cudaEventDestroy(ev);
        if (r.ev_raw) cudaEventDestroy(r.ev_raw);
        if (r.ev_lists) cudaEventDestroy(r.ev_lists);
    }
    if (c->ev_probe) cudaEventDestroy(c->ev_probe);
    if (c->f64_stream) cudaStreamDestroy(c->f64_stream);
    if (c->ev_block) cudaEventDestroy(c->ev_block);
    if (c->ev_poll) cudaEventDestroy(c->ev_poll);
    if (c->list_stream) cudaStreamDestroy(c->list_stream);
    if (c->ev_h2d) cudaEventDestroy(c->ev_h2d);
    if (c->ev_ref) cudaEventDestroy(c->ev_ref);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
    delete c;
}

const char* pmm_last_error(const pmm_ctx* c) { return c ? c->err.c_str() : g_create_error.c_str(); }

int pmm_set_option(pmm_ctx* c, const char* key, const char* value)
{
    if (!c || !key || !value) return PMM_ERR_INVALID;
    const std::string k(key);
    if (k == "stream") {
        const std::string sv(value);
        if (sv == "own") c->stream = c->own_stream;
        else if (sv == "default") c->stream = nullptr;                       // the legacy default stream
        else c->stream = reinterpret_cast<cudaStream_t>(strtoull(value, nullptr, 0));
        return PMM_OK;
    }
    if (k == "priority") {
        // rank of this context's kernels among the contexts sharing the GPU: 0 = first in line (highest CUDA stream
        // priority), larger = later.  The kernels are persistent (one launch fills the GPU), so the order only decides
        // whose blocks take the slots another kernel's tail frees -- e.g. the double re-run of tile k before the float
        // pass of tile k+2 when a batch is cut into tiles that run on several contexts (pairhmm/client/PairHMMWorker).
        const int rank = atoi(value);
        if (rank < 0 || rank > 64) return c->fail(PMM_ERR_INVALID, "priority rank out of range");
        cudaSetDevice(c->device);
        int least = 0, greatest = 0;
        PMM_CUDA(c, cudaDeviceGetStreamPriorityRange(&least, &greatest));        // numerically: greatest <= least
        const int prio = std::min(least, greatest + rank);
        PMM_CUDA(c, cudaStreamSynchronize(c->own_stream));
        PMM_CUDA(c, cudaStreamSynchronize(c->f64_stream));
        cudaStream_t ns = nullptr, nd = nullptr;
        cudaError_t e = cudaStreamCreateWithPriority(&ns, cudaStreamNonBlocking, prio);
        if (e == cudaSuccess && (e = create_f64_stream(&nd, prio)) != cudaSuccess) cudaStreamDestroy(ns);
        if (e != cudaSuccess) return c->fail_cuda(e, "priority streams");
        const bool was_own = c->stream == c->own_stream;
        cudaStreamDestroy(c->own_stream); cudaStreamDestroy(c->f64_stream);
        c->own_stream = ns; c->f64_stream = nd;
        if (was_own) c->stream = ns;
        return PMM_OK;
    }
    if (k == "tasks_per_warp") {
        const int v = atoi(value);
        if (v < 1 || v > 64) return c->fail(PMM_ERR_INVALID, "tasks_per_warp out of range");
        c->plan_opt.tasks_per_warp = v;
        return PMM_OK;
    }
    if (k == "small_job_widening") {
        const std::string v(value);
        if (v != "0" && v != "1" && v != "on" && v != "off") return c->fail(PMM_ERR_INVALID, "small_job_widening is \"on\" or \"off\"");
        c->plan_opt.widening = v == "1" || v == "on";
        return PMM_OK;
    }
    if (k == "run_tiers") {
        int d = -1, share = kRunTierShare, top = kRunTierTop;
        if (std::sscanf(value, "%d,%d,%d", &d, &share, &top) < 1 || d < 0 || d > 64 || share < 1 || share > 100 || top < 1 || top > 64)
            return c->fail(PMM_ERR_INVALID, "run_tiers is \"depth[,share[,top]]\", depth 0..64, share 1..100, top 1..64");
        c->plan_opt.tiers = RunTiers{d, share, top};
        return PMM_OK;
    }
    if (k == "f64_tasks_per_warp" || k == "f64_max_run") {
        const int v = atoi(value);
        if (v < 1 || v > 64) return c->fail(PMM_ERR_INVALID, k + " out of range (1..64)");
        (k == "f64_max_run" ? c->f64_max_run : c->f64_tasks_per_warp) = v;
        return PMM_OK;
    }
    if (k == "overlap") {
        const std::string v(value);
        if (v != "0" && v != "1" && v != "on" && v != "off") return c->fail(PMM_ERR_INVALID, "overlap is \"on\" or \"off\"");
        c->overlap = v == "1" || v == "on";
        return PMM_OK;
    }
    if (k == "mode") {
        const std::string v(value);
        if (v != "exact" && v != "fast") return c->fail(PMM_ERR_INVALID, "mode is \"exact\" or \"fast\"");
        c->fast = v == "fast";
        return PMM_OK;
    }
    if (k == "guard") {
        const float g = (float)atof(value);
        if (!(g >= 0.0f && g < 1.0f)) return c->fail(PMM_ERR_INVALID, "guard must be in [0, 1)");
        c->guard = g;
        return PMM_OK;
    }
    if (k == "sync") {
        const std::string v = value;
        if (v != "spin" && v != "block" && v != "hybrid" && v != "auto") return c->fail(PMM_ERR_INVALID, "sync is \"spin\", \"block\", \"hybrid\" or \"auto\"");
        c->block_sync = v == "block" || v == "hybrid";
        c->spin_us = v == "hybrid" ? 60 : 0;
        c->auto_sync = v == "auto";
        return PMM_OK;
    }
    if (k == "force_variant") {
        int K = 0, W = 0;
        if (sscanf(value, "%d,%d", &K, &W) != 2 || (K > 0 && !forward_f32_has_variant(K, W)))
            return c->fail(PMM_ERR_INVALID, "force_variant wants \"K,W\" of an instantiated float kernel, \"0,0\" (planner's choice) or \"-1,0\" (no consolidation of rare variants)");
        c->plan_opt.force = K > 0 ? Variant{K, W, false} : Variant{0, 0, false};
        c->plan_opt.keep_all_variants = K < 0;
        return PMM_OK;
    }
    return c->fail(PMM_ERR_INVALID, "unknown option " + k);
}

int pmm_stage_flat(pmm_ctx* c, uint32_t num_read, const uint32_t* read_off,
                   const uint8_t* bases, const uint8_t* q, const uint8_t* i, const uint8_t* d, const uint8_t* cc,
                   uint32_t num_hap, const uint32_t* hap_off, const uint8_t* hap_bases,
                   uint32_t num_region, const pmm_region_t* regions)
{
    return guarded(c, [&]() -> int {
        if (!c) return PMM_ERR_INVALID;
        if (!bases || !q || !i || !d || !cc || !hap_bases) return c->fail(PMM_ERR_INVALID, "null track");
        if (!read_off || !hap_off || !num_read || !num_hap) return c->fail(PMM_ERR_INVALID, "empty job");
        // before source_from_flat takes offsets relative to the first ones
        if (read_off[num_read] < read_off[0] || hap_off[num_hap] < hap_off[0]) return c->fail(PMM_ERR_INVALID, "offsets not ascending");
        for (uint32_t k = 0; k < num_read; ++k) if (read_off[k + 1] < read_off[k]) return c->fail(PMM_ERR_INVALID, "offsets not ascending");
        for (uint32_t k = 0; k < num_hap; ++k) if (hap_off[k + 1] < hap_off[k]) return c->fail(PMM_ERR_INVALID, "offsets not ascending");
        const uint8_t* const tracks[5] = {bases, q, i, d, cc};
        source_from_flat(c->src, num_read, read_off, tracks, num_hap, hap_off, hap_bases, num_region, regions);
        return stage(c, c->src);
    });
}

int pmm_launch(pmm_ctx* c)
{
    if (!c) return PMM_ERR_INVALID;
    if (!c->staged) return c->fail(PMM_ERR_STATE, "pmm_launch before pmm_stage_*");
    const StagedJob& j = c->job;
    if (c->fast && c->d_tiny_tasks.cap < sizeof(Task) * j.pairs) return c->fail(PMM_ERR_STATE, "mode changed to fast after pmm_stage_*: stage the job again");
    cudaSetDevice(c->device);
    cudaStream_t s = c->stream, sd = c->f64_stream;
    // This launch takes the other result set: the previous launch's double re-run may still be using its own.
    ResultSet& prev = c->rs[c->cur];
    c->cur ^= 1;
    ResultSet& R = c->rs[c->cur];
    // control words, hot ones on their own 128-byte lines: [0] fallback count, [1] flush count, [2] re-check count,
    // [3] tasks of the double re-run, [4] fallback slots handed out, [kCtrlHist ..) and [kCtrlClassCursor ..) the counting
    // sort of those tasks, [kCtrlCursors + 32 k] work-queue cursor of launch k
    uint32_t* ctrl = static_cast<uint32_t*>(R.d_ctrl.p);
    uint32_t launches = 0;
    c->launched = false; c->have_raw = false; c->have_lists = false;
    // the launch before the previous one used this set: its copies out of d_raw, d_ctrl and the fallback list (which
    // follow its double re-run) must be over (no-ops the first times)
    PMM_CUDA(c, cudaStreamWaitEvent(s, R.ev_raw, 0));
    PMM_CUDA(c, cudaStreamWaitEvent(s, R.ev_lists, 0));
    PMM_CUDA(c, cudaEventRecord(R.ev[0], s));
    PMM_CUDA(c, cudaMemsetAsync(ctrl, 0, sizeof(uint32_t) * kCtrlWords, s));

    ForwardArgs a{};
    a.read_blob = section<uint8_t>(c->d_in.p, j.at.rblob);
    a.reads = section<ReadDesc>(c->d_in.p, j.at.rdesc);
    a.stream = static_cast<uint8_t*>(c->d_stream.p) + kStreamFrontPad;
    a.spos = section<uint32_t>(c->d_in.p, j.at.spos);
    a.tab = c->dtab;
    a.scratch = c->d_scratch.p;
    a.scratch_stride = j.max_hap_len + 8;

    // ---- row parameters, once per read (the reference recomputes them per pair) --------------------------------
    a.params = static_cast<float*>(c->d_params.p);
    PMM_CUDA(c, launch_read_params(a.read_blob, a.reads, section<GroupDesc>(c->d_in.p, j.at.groups), j.num_groups,
                                   c->dtab, static_cast<float*>(c->d_params.p), s));
    ++launches;

    // ---- float pass, one launch per (K, W) variant present in the job; results below 1e-28f are appended to the
    //      fallback list by the kernel itself (PairHMMWorker.cpp:176) ----------------------------------------------
    if (j.segs.size() > 100) return c->fail(PMM_ERR_INVALID, "too many kernel variants in one job");
    // fast mode: results within the guard band around the threshold are re-run by an exact kernel before the decision
    // is taken, so the decision (and the float value of those pairs) is the reference's, bit for bit
    const float thr = 1e-28f;
    FallbackQueue fq{ctrl + 0, (uint32_t)j.pairs,
                     c->fast ? thr * (1.0f - c->guard) : thr, c->fast ? thr * (1.0f + c->guard) : thr,
                     static_cast<Task*>(c->d_tiny_tasks.p), ctrl + 2};
    uint32_t cursor = kCtrlCursors;
    for (const LaunchSeg& seg : j.segs) {
        a.inity = c->d_iyf.p;
        a.tasks = section<Task>(c->d_in.p, j.at.tasks) + seg.task_first;
        a.ntasks = seg.task_count; a.ntasks_dev = nullptr;
        a.counter = ctrl + cursor; cursor += 32;
        a.out = R.d_raw.p;
        const ForwardKernel* fk = forward_f32_variant(seg.v.K, seg.v.W, seg.v.striped, c->fast);
        const int per_sm = fk ? fk->ctas_per_sm() : 0;
        if (per_sm <= 0) return c->fail(PMM_ERR_INVALID, "kernel variant unavailable");
        const int ctas = (int)std::min<uint64_t>((seg.task_count + kWarpsPerCta - 1) / kWarpsPerCta, (uint64_t)c->sm_count * per_sm);
        PMM_CUDA(c, fk->launch(a, fq, ctas, s));
        ++launches;
    }
    if (c->fast) {
        // ---- exact re-check of the guard band (normally a handful of pairs, often none) -----------------------------
        a.tasks = static_cast<Task*>(c->d_tiny_tasks.p); a.ntasks = 0; a.ntasks_dev = ctrl + 2;
        a.counter = ctrl + cursor; cursor += 32;
        fq.lo = fq.hi = thr;
        PMM_CUDA(c, recheck_f32_variant().launch(a, fq, c->sm_count * std::max(1, recheck_f32_variant().ctas_per_sm()), s));
        ++launches;
    }
    PMM_CUDA(c, cudaEventRecord(R.ev[1], s));
    // The raw floats are final now: copy them back on the copy stream while the double pass runs, so that a fetch can
    // take log10f of them (host libm) under it.
    const HostOut ho = host_out(R, j.pairs);
    PMM_CUDA(c, cudaStreamWaitEvent(c->copy_stream, R.ev[1], 0));
    PMM_CUDA(c, cudaMemcpyAsync(ho.raw, R.d_raw.p, sizeof(float) * j.pairs, cudaMemcpyDeviceToHost, c->copy_stream));
    PMM_CUDA(c, cudaEventRecord(R.ev_raw, c->copy_stream));

    // ---- double re-run (PairHMMWorker.cpp:176-184): the results below the threshold become tasks, the failing haplotypes
    //      of a read together; their number is only known on the device.  On its own stream: the next launch's float pass
    //      (this stream) starts as soon as this one's is over and runs next to it ------------------------------------------
    PMM_CUDA(c, cudaStreamWaitEvent(sd, R.ev[1], 0));
    const ForwardKernel* dk = forward_f64_variant(j.f64_rows, j.f64_striped);      // one of kF64Rows: never null
    const int f64_ctas = c->sm_count * std::max(1, dk->ctas_per_sm());
    FallbackBuild fb{};
    fb.raw = static_cast<float*>(R.d_raw.p);
    fb.regions = section<RegionDesc>(c->d_in.p, j.at.regions);
    fb.reads = a.reads;
    fb.num_region = j.num_region; fb.num_rows = j.num_rows;
    fb.threshold = thr;
    fb.ctrl = ctrl;
    fb.tasks = static_cast<Task*>(R.d_fb_tasks.p);
    fb.out_index = static_cast<uint32_t*>(R.d_fb_idx.p);
    fb.hap_list = static_cast<uint32_t*>(R.d_fb_hap.p);
    fb.row_slot = static_cast<uint32_t*>(R.d_fb_rows.p);
    fb.spos = a.spos;
    fb.max_hap_len = j.max_hap_len;
    fb.capacity = (uint32_t)j.pairs;
    fb.single_stripe_rows = 32u * (uint32_t)j.f64_rows;
    fb.target_tasks = (uint32_t)(f64_ctas * kWarpsPerCta * c->f64_tasks_per_warp);
    fb.max_run = (uint32_t)c->f64_max_run;
    PMM_CUDA(c, launch_build_fallback(fb, c->sm_count, sd));
    launches += 2;
    a.inity = c->d_iyd.p; a.out = R.d_dres.p; a.tasks = fb.tasks; a.hap_list = fb.hap_list;
    a.ntasks = 0; a.ntasks_dev = ctrl + 3; a.counter = ctrl + cursor; cursor += 32;
    a.tiny_threshold = ldexp(1.0, -800); a.tiny_count = ctrl + 1;
    a.scratch = c->d_scratch64.p;
    PMM_CUDA(c, dk->launch(a, FallbackQueue{}, f64_ctas, sd));
    ++launches;
    PMM_CUDA(c, cudaEventRecord(R.ev[2], sd));
    // What is queued on the launch stream from here on (the next launch, an event of the caller's) comes after the
    // PREVIOUS launch's double re-run: consecutive launches overlap by one pass, no further, and a pair of events around
    // each pmm_launch of a steady sequence brackets exactly one float pass and one double re-run.
    PMM_CUDA(c, cudaStreamWaitEvent(s, (c->overlap ? prev : R).ev[2], 0));
    // The length of the fallback list is only known on the device.  Copy the control words and a first slice of the list
    // (an eighth of the pairs) back right behind the double pass, so that the common case needs no further round trip;
    // the rest, if any, follows in the fetch.
    c->spec = (uint32_t)std::min<uint64_t>(j.pairs, std::max<uint64_t>(1024, j.pairs / 8));
    cudaStream_t ls = c->list_stream;                           // not a kernels' stream: the next job need not wait for these
    PMM_CUDA(c, cudaStreamWaitEvent(ls, R.ev[2], 0));
    PMM_CUDA(c, cudaMemcpyAsync(ho.ctrl, R.d_ctrl.p, 12, cudaMemcpyDeviceToHost, ls));
    PMM_CUDA(c, cudaMemcpyAsync(ho.idx, R.d_fb_idx.p, sizeof(uint32_t) * c->spec, cudaMemcpyDeviceToHost, ls));
    PMM_CUDA(c, cudaMemcpyAsync(ho.dres, R.d_dres.p, sizeof(double) * c->spec, cudaMemcpyDeviceToHost, ls));
    PMM_CUDA(c, cudaEventRecord(R.ev_lists, ls));
    c->stats.kernel_launches = launches;
    c->launched = true;
    return PMM_OK;
}

int pmm_join(pmm_ctx* c)
{
    if (!c) return PMM_ERR_INVALID;
    if (!c->launched) return PMM_OK;
    cudaSetDevice(c->device);
    PMM_CUDA(c, cudaStreamWaitEvent(c->stream, c->R().ev[2], 0));
    return PMM_OK;
}

int pmm_sync(pmm_ctx* c)
{
    if (!c) return PMM_ERR_INVALID;
    cudaSetDevice(c->device);
    PMM_CUDA(c, cudaStreamSynchronize(c->stream));
    PMM_CUDA(c, cudaStreamSynchronize(c->f64_stream));
    PMM_CUDA(c, cudaStreamSynchronize(c->copy_stream));
    PMM_CUDA(c, cudaStreamSynchronize(c->list_stream));
    if (c->launched) {
        cudaEventElapsedTime(&c->stats.ms_f32, c->R().ev[0], c->R().ev[1]);
        cudaEventElapsedTime(&c->stats.ms_fallback, c->R().ev[1], c->R().ev[2]);
    }
    return PMM_OK;
}

// Wait for everything queued on one of the context's streams.  A caller with one context per core spins (lowest latency);
// the pool, which runs several contexts per GPU from as many host threads, can sleep on a blocking event so that the
// waiting threads do not take the cores the packing and log10 work of the other contexts needs.
// "auto": a spinning wait is the fastest (no wake-up), but every spinner holds a core.  The first few waiting threads
// of the process spin, the rest sleep -- a host with one or two caller threads gets the latency, a host with dozens (or a
// box with a process per GPU) keeps its cores for the packing and log10 work.
static std::atomic<int> g_spinners{0};
static int spinner_budget()
{
    static const int b = [] { const unsigned hw = std::thread::hardware_concurrency(); return (int)std::max(1u, hw / 16); }();
    return b;
}

static cudaError_t wait_stream(pmm_ctx* c, cudaStream_t st)
{
    if (c->auto_sync) {
        // Whoever finds a spinner's place free takes it (the earliest waiter, i.e. the job that finishes first); the others
        // nap and look again -- for the event and for a free place -- so a waiter is promoted as soon as the one ahead of it
        // is done, and a sleeping thread never costs more than a wake-up of a few tens of microseconds.
        cudaError_t e = cudaEventRecord(c->ev_poll, st);
        if (e != cudaSuccess) return e;
        for (;;) {
            if (g_spinners.fetch_add(1, std::memory_order_relaxed) < spinner_budget()) {
                e = cudaEventSynchronize(c->ev_poll);
                g_spinners.fetch_sub(1, std::memory_order_relaxed);
                return e;
            }
            g_spinners.fetch_sub(1, std::memory_order_relaxed);
            e = cudaEventQuery(c->ev_poll);
            if (e != cudaErrorNotReady) return e;
            std::this_thread::sleep_for(std::chrono::microseconds(25));
        }
    }
    if (!c->block_sync) return cudaStreamSynchronize(st);
    cudaError_t e = cudaEventRecord(c->ev_block, st);
    if (e != cudaSuccess) return e;
    if (c->spin_us > 0) {
        // hybrid: what is about to finish is caught without a wake-up, what takes long does not hold a core
        const auto until = std::chrono::steady_clock::now() + std::chrono::microseconds(c->spin_us);
        do {
            e = cudaEventQuery(c->ev_block);
            if (e != cudaErrorNotReady) return e;
        } while (std::chrono::steady_clock::now() < until);
    }
    return cudaEventSynchronize(c->ev_block);
}

// The raw floats of the last launch are in h_out (copied by pmm_launch on the copy stream; the double pass may still run).
static int ensure_raw(pmm_ctx* c)
{
    if (!c->launched) return c->fail(PMM_ERR_STATE, "fetch before pmm_launch");
    if (c->have_raw) return PMM_OK;
    cudaSetDevice(c->device);
    PMM_CUDA(c, wait_stream(c, c->copy_stream));
    c->have_raw = true;
    return PMM_OK;
}

// The control words and the whole fallback list of the last launch are in h_out.  Every fetch_* of one launch shares
// these copies: nothing is transferred twice.
static int ensure_lists(pmm_ctx* c)
{
    if (!c->launched) return c->fail(PMM_ERR_STATE, "fetch before pmm_launch");
    if (c->have_lists) return PMM_OK;
    cudaSetDevice(c->device);
    cudaStream_t s = c->list_stream;
    const HostOut o = host_out(c->R(), c->job.pairs);
    PMM_CUDA(c, wait_stream(c, s));
    const uint32_t nfb = o.ctrl[0], spec = c->spec;
    uint64_t d2h = 12 + sizeof(float) * c->job.pairs + (sizeof(uint32_t) + sizeof(double)) * spec;
    if (nfb > spec) {
        PMM_CUDA(c, cudaMemcpyAsync(o.idx + spec, static_cast<uint32_t*>(c->R().d_fb_idx.p) + spec, sizeof(uint32_t) * (nfb - spec), cudaMemcpyDeviceToHost, s));
        PMM_CUDA(c, cudaMemcpyAsync(o.dres + spec, static_cast<double*>(c->R().d_dres.p) + spec, sizeof(double) * (nfb - spec), cudaMemcpyDeviceToHost, s));
        PMM_CUDA(c, cudaEventRecord(c->R().ev_lists, s));
        PMM_CUDA(c, wait_stream(c, s));
        d2h += (sizeof(uint32_t) + sizeof(double)) * (nfb - spec);
    }
    c->stats.fallback_pairs = nfb; c->stats.flush_pairs = o.ctrl[1]; c->stats.recheck_pairs = o.ctrl[2]; c->stats.d2h_bytes = d2h;
    cudaEventElapsedTime(&c->stats.ms_f32, c->R().ev[0], c->R().ev[1]);
    cudaEventElapsedTime(&c->stats.ms_fallback, c->R().ev[1], c->R().ev[2]);
    c->have_lists = true;
    return PMM_OK;
}

// (double)(log10f(v) - log10f(2^120)), float subtraction (PairHMMWorker.cpp:190); host libm on purpose
static void log10_of_raw(const float* raw, uint64_t n, double* out)
{
    const float licf = host_tables().log10_ic_f;
    host_parallel_for(n, 1 << 13, [&](uint64_t a, uint64_t b) { for (uint64_t k = a; k < b; ++k) out[k] = (double)(log10f(raw[k]) - licf); });
}
// log10(d) - log10(2^1020) for the pairs that fell back (PairHMMWorker.cpp:184)
static int log10_of_fallback(const uint32_t* fb_index, const double* fb_value, uint64_t n_fb, uint64_t n, double* out)
{
    const double licd = host_tables().log10_ic_d;
    for (uint64_t k = 0; k < n_fb; ++k) {
        if (fb_index[k] >= n) return PMM_ERR_INVALID;
        out[fb_index[k]] = log10(fb_value[k]) - licd;
    }
    return PMM_OK;
}

int pmm_fetch_raw(pmm_ctx* c, float* out_raw, uint64_t cap)
{
    if (!c || !out_raw) return PMM_ERR_INVALID;
    if (cap < c->job.pairs) return c->fail(PMM_ERR_INVALID, "output buffer too small");
    auto t0 = std::chrono::steady_clock::now();
    int rc = ensure_raw(c);
    if (rc) return rc;
    memcpy(out_raw, host_out(c->R(), c->job.pairs).raw, sizeof(float) * c->job.pairs);
    c->stats.ms_fetch = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    return PMM_OK;
}

int pmm_fetch_fallback_mask(pmm_ctx* c, uint8_t* mask, uint64_t cap)
{
    if (!c || !mask) return PMM_ERR_INVALID;
    if (cap < c->job.pairs) return c->fail(PMM_ERR_INVALID, "mask buffer too small");
    int rc = ensure_lists(c);
    if (rc) return rc;
    memset(mask, 0, c->job.pairs);
    const HostOut o = host_out(c->R(), c->job.pairs);
    for (uint32_t k = 0; k < o.ctrl[0]; ++k) mask[o.idx[k]] = 1;
    return PMM_OK;
}

int pmm_host_finish_log10(const float* raw, uint64_t n, const uint32_t* fb_index, const double* fb_value, uint64_t n_fb, double* out)
{
    if (!out || (n && !raw) || (n_fb && (!fb_index || !fb_value))) return PMM_ERR_INVALID;
    log10_of_raw(raw, n, out);
    return log10_of_fallback(fb_index, fb_value, n_fb, n, out);
}

// The final doubles of the last launch: log10f of the raw floats is taken while the double pass is still running.
int pmm_fetch_log10(pmm_ctx* c, double* out, uint64_t cap, uint64_t* n_fallback)
{
    if (!c || !out) return PMM_ERR_INVALID;
    if (cap < c->job.pairs) return c->fail(PMM_ERR_INVALID, "output buffer too small");
    auto t0 = std::chrono::steady_clock::now();
    int rc = ensure_raw(c);
    if (rc) return rc;
    const HostOut o = host_out(c->R(), c->job.pairs);
    log10_of_raw(o.raw, c->job.pairs, out);
    if ((rc = ensure_lists(c))) return rc;
    if (log10_of_fallback(o.idx, o.dres, o.ctrl[0], c->job.pairs, out) != PMM_OK) return c->fail(PMM_ERR_CUDA, "fallback index out of range");
    if (n_fallback) *n_fallback = o.ctrl[0];
    c->stats.ms_fetch = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    return PMM_OK;
}

int pmm_fetch_fallback(pmm_ctx* c, uint32_t* index, double* value, uint64_t cap, uint64_t* count)
{
    if (!c || !count) return PMM_ERR_INVALID;
    int rc = ensure_lists(c);
    if (rc) return rc;
    const HostOut o = host_out(c->R(), c->job.pairs);
    const uint32_t nfb = o.ctrl[0];
    *count = nfb;
    if (!index && !value) return PMM_OK;
    if (!index || !value || cap < nfb) return c->fail(PMM_ERR_INVALID, "fallback buffers too small");
    memcpy(index, o.idx, sizeof(uint32_t) * nfb);
    memcpy(value, o.dres, sizeof(double) * nfb);
    return PMM_OK;
}

int pmm_stage_serialized(pmm_ctx* c, const void* reads_ser, uint64_t reads_bytes, const void* haps_ser,
                         uint64_t haps_bytes, int* num_read, int* num_hap)
{
    return guarded(c, [&]() -> int {
        if (!c) return PMM_ERR_INVALID;
        const int rc = source_from_serialized(c, reads_ser, reads_bytes, haps_ser, haps_bytes, num_read, num_hap);
        return rc ? rc : stage(c, c->src);
    });
}

int pmm_get_stats(const pmm_ctx* c, pmm_stats_t* out)
{
    if (!c || !out) return PMM_ERR_INVALID;
    *out = c->stats;
    return PMM_OK;
}

int pmm_forward_raw_serialized(pmm_ctx* c, const void* reads_ser, uint64_t reads_bytes, const void* haps_ser,
                               uint64_t haps_bytes, float* out_raw, uint64_t cap, int* num_read, int* num_hap)
{
    return guarded(c, [&]() -> int {
        if (!c || !out_raw) return PMM_ERR_INVALID;
        return stage_launch_fetch(c, source_from_serialized(c, reads_ser, reads_bytes, haps_ser, haps_bytes, num_read, num_hap),
                                  [&] { return pmm_fetch_raw(c, out_raw, cap); });
    });
}

int pmm_forward_log10_serialized(pmm_ctx* c, const void* reads_ser, uint64_t reads_bytes, const void* haps_ser,
                                 uint64_t haps_bytes, double* out, uint64_t cap, int* num_read, int* num_hap,
                                 uint64_t* n_fallback)
{
    return guarded(c, [&]() -> int {
        if (!c || !out) return PMM_ERR_INVALID;
        return stage_launch_fetch(c, source_from_serialized(c, reads_ser, reads_bytes, haps_ser, haps_bytes, num_read, num_hap),
                                  [&] { return pmm_fetch_log10(c, out, cap, n_fallback); });
    });
}

int pmm_forward_log10(pmm_ctx* c, const pmm_read_t* reads, int num_read, const pmm_hap_t* haps, int num_hap,
                      double* out, uint64_t* n_fallback)
{
    return guarded(c, [&]() -> int {
        if (!c || !reads || !haps || !out || num_read <= 0 || num_hap <= 0) return c ? c->fail(PMM_ERR_INVALID, "bad arguments") : PMM_ERR_INVALID;
        return stage_launch_fetch(c, source_from_structs(c, reads, num_read, haps, num_hap),
                                  [&] { return pmm_fetch_log10(c, out, (uint64_t)num_read * num_hap, n_fallback); });
    });
}

int pmm_forward_log10_testcases(pmm_ctx* c, const pmm_testcase_t* tc, uint64_t n, double* out, uint64_t* n_fallback)
{
    return guarded(c, [&]() -> int {
        if (!c) return PMM_ERR_INVALID;
        if (!tc || !out || !n) return c->fail(PMM_ERR_INVALID, "bad arguments");
        if (n >= (1ull << 31)) return c->fail(PMM_ERR_INVALID, "more than 2^31 pairs in one batch: split it");
        return stage_launch_fetch(c, source_from_testcases(c, tc, n), [&] { return pmm_fetch_log10(c, out, n, n_fallback); });
    });
}

int pmm_plan_flat(uint32_t num_read, const uint32_t* read_off, uint32_t num_hap, const uint32_t* hap_off,
                  uint32_t num_region, const pmm_region_t* regions, int sm_count, int tasks_per_warp,
                  pmm_task_info_t* out, uint64_t capacity, uint64_t* num_tasks)
{
    return guarded(nullptr, [&]() -> int {
        PlanOptions opt = plan_defaults();
        opt.tasks_per_warp = tasks_per_warp;
        Plan plan; std::string perr;
        int rc = plan_job(num_read, read_off, num_hap, hap_off, num_region, regions, sm_count, opt, plan, perr);
        if (rc) { g_create_error = perr; return rc; }
        if (num_tasks) *num_tasks = plan.tasks.size();
        if (!out) return PMM_OK;
        if (capacity < plan.tasks.size()) { g_create_error = "task buffer too small"; return PMM_ERR_INVALID; }
        for (const LaunchSeg& seg : plan.segs)
            for (uint32_t k = seg.task_first; k < seg.task_first + seg.task_count; ++k) {
                const Task& t = plan.tasks[k];
                pmm_task_info_t& o = out[k];
                for (int z = 0; z < 4; ++z) { o.read[z] = t.read[z]; o.out_base[z] = t.out_base[z]; }
                o.hap_first = t.hap_first; o.num_hap = t.nhaps; o.num_read = t.nreads;
                o.rows_per_lane = (uint32_t)seg.v.K; o.lanes_per_read = (uint32_t)seg.v.W; o.striped = seg.v.striped ? 1u : 0u;
            }
        return PMM_OK;
    });
}

int pmm_host_table(int which, void* out, uint64_t capacity_bytes)
{
    const HostTables& t = host_tables();
    const void* src = nullptr; size_t n = 0;
    switch (which) {
        case 0: src = t.ph2pr_f; n = sizeof t.ph2pr_f; break;
        case 1: src = t.m2m_f;   n = sizeof t.m2m_f;   break;
        case 2: src = t.ph2pr_d; n = sizeof t.ph2pr_d; break;
        case 3: src = t.m2m_d;   n = sizeof t.m2m_d;   break;
        case 4: src = &t.log10_ic_f; n = sizeof(float); break;
        case 5: src = &t.log10_ic_d; n = sizeof(double); break;
        default: return PMM_ERR_INVALID;
    }
    if (!out || capacity_bytes < n) return PMM_ERR_INVALID;
    memcpy(out, src, n);
    return PMM_OK;
}

int pmm_measure_fp32_peak(pmm_ctx* c, double* lane_instr_per_s, double* sm_mhz)
{
    if (!c || !lane_instr_per_s) return PMM_ERR_INVALID;
    cudaSetDevice(c->device);
    const int ctas = c->sm_count * 8, iters = 500;
    PMM_CUDA(c, c->d_probe.reserve(sizeof(float) * ctas * 256));
    float* sink = static_cast<float*>(c->d_probe.p);
    const int rc = probe_rate(c, [&](int n) { return launch_fp32_probe(sink, n, ctas, c->stream); }, 25, iters,
                              (double)ctas * 256 * iters * 512.0, lane_instr_per_s);
    if (rc) return rc;
    if (sm_mhz) *sm_mhz = *lane_instr_per_s / ((double)c->sm_count * 128.0) * 1e-6;   // lower bound: assumes 128 lanes/clk/SM fully used
    return PMM_OK;
}

int pmm_get_timeline(pmm_ctx* c, pmm_timeline_t* out)
{
    if (!c || !out) return PMM_ERR_INVALID;
    if (!c->launched) return c->fail(PMM_ERR_STATE, "pmm_get_timeline before pmm_launch");
    cudaSetDevice(c->device);
    PMM_CUDA(c, cudaEventSynchronize(c->R().ev[2]));
    float a = 0, b = 0, d = 0;
    PMM_CUDA(c, cudaEventElapsedTime(&a, c->ev_ref, c->R().ev[0]));
    PMM_CUDA(c, cudaEventElapsedTime(&b, c->ev_ref, c->R().ev[1]));
    PMM_CUDA(c, cudaEventElapsedTime(&d, c->ev_ref, c->R().ev[2]));
    out->ref_host_s = c->ref_host_s;
    out->kernels_start_s = a * 1e-3; out->f32_end_s = b * 1e-3; out->kernels_end_s = d * 1e-3;
    return PMM_OK;
}

int pmm_measure_fp64_peak(pmm_ctx* c, double* lane_instr_per_s)
{
    if (!c || !lane_instr_per_s) return PMM_ERR_INVALID;
    cudaSetDevice(c->device);
    const int ctas = c->sm_count * 8, iters = 60;
    PMM_CUDA(c, c->d_probe.reserve(sizeof(double) * ctas * 256));
    double* sink = static_cast<double*>(c->d_probe.p);
    return probe_rate(c, [&](int n) { return launch_fp64_probe(sink, n, ctas, c->stream); }, 5, iters,
                      (double)ctas * 256 * iters * 512.0, lane_instr_per_s);
}

}  // extern "C"
