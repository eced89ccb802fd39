// pmm_pool.cpp -- host-side work queue over the GPUs of one box (SURVEY.md section 8e).
//
// Read x haplotype pairs are independent and nothing is reduced, so multi-GPU is a partition of whole regions with
// no collective: the pool owns `contexts_per_device` engine contexts (pmm_ctx, each with its own stream and pinned
// staging buffers) on every device it was given and one feeder thread per pair of contexts.  Jobs go into one queue
// served by generation (a run of consecutive tickets) and, inside a generation, largest first (the skewed length
// distribution of configs 4/5 leaves the small jobs to fill the tail); a feeder takes the next job, stages it,
// launches and fetches it through the same C ABI a single-GPU caller uses, always with a second job already queued on
// the GPU behind the one it is waiting for.  This is the piece that stands where the reference has Blaze's per-accelerator task queue
// and the FPGA processing-unit balancer (/root/reference/pairhmm/interface/PairHMMFpgaInterface.cpp:67-170).
#include "../../include/pairhmm_cuda.h"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <queue>
#include <string>
#include <thread>
#include <vector>

namespace {

struct Job {
    uint64_t ticket = 0, cells = 0, pairs = 0, generation = 0;
    // flat layout, borrowed from the caller until pmm_pool_wait returns
    uint32_t num_read = 0, num_hap = 0, num_region = 0;
    const uint32_t* read_off = nullptr; const uint8_t* tr[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    const uint32_t* hap_off = nullptr; const uint8_t* hap = nullptr;
    const pmm_region_t* regions = nullptr;
    pmm_region_t one_region{};
    double* out = nullptr; uint64_t out_capacity = 0;
    // completion
    int rc = PMM_OK; std::string err; uint64_t n_fallback = 0; int device = -1; bool done = false;
};

// Order of service: by generation (a run of consecutive tickets), inside a generation the largest job first.  Largest
// first is what balances a bounded set of jobs (the small ones fill the tail), but as the only key it starves the small
// jobs of a continuous stream behind ever newer large ones -- with eight GPUs draining the queue that stalled a caller
// waiting for its oldest ticket every ~50 ms on all devices at once (profiles/r02_pool_timeline_n8_before.jsonl).
struct JobOrder {
    bool operator()(const Job* a, const Job* b) const            // priority_queue: "less" = served later
    {
        if (a->generation != b->generation) return a->generation > b->generation;
        if (a->cells != b->cells) return a->cells < b->cells;
        return a->ticket > b->ticket;
    }
};

}  // namespace

struct pmm_pool {
    std::vector<pmm_ctx*> ctxs;
    std::vector<int> ctx_device;
    std::vector<std::thread> feeders;
    std::mutex mu;
    std::condition_variable cv_work, cv_done;
    std::priority_queue<Job*, std::vector<Job*>, JobOrder> queue;
    std::map<uint64_t, Job*> jobs;                 // every submitted, not yet collected job
    uint64_t next_ticket = 1;
    bool stopping = false;
    std::string err;
    std::vector<uint64_t> cells_per_device, jobs_per_device;
    int n_devices = 0;
    std::vector<int> devices;
    bool tracing = false;               // pmm_pool_trace: one record per GPU job
    std::vector<pmm_pool_trace_t> trace;
    std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
};

static thread_local std::string g_pool_error;      // errors of calls without a pool, and the text pmm_pool_last_error hands out

static double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

// One GPU job of a feeder: the submitted job it serves, where it is in its life, and the host times of the trace.
struct Flight {
    Job* job = nullptr;
    bool active = false;                // staged and launched, results not yet fetched
    int rc = PMM_OK;                    // of staging and launch
    double t_take = 0, t_staged = 0, t_launched = 0;
};

// Stage and launch; the kernels run while the caller does something else.
static void start_job(pmm_ctx* c, Flight& f)
{
    const Job* j = f.job;
    f.rc = pmm_stage_flat(c, j->num_read, j->read_off, j->tr[0], j->tr[1], j->tr[2], j->tr[3], j->tr[4],
                          j->num_hap, j->hap_off, j->hap, j->num_region, j->regions);
    f.t_staged = now_s();
    if (f.rc == PMM_OK) f.rc = pmm_launch(c);
    f.t_launched = now_s();
}

// Fetch the results into the caller's buffer and record the job's status.
static void finish_job(pmm_ctx* c, const Flight& f)
{
    Job* j = f.job;
    uint64_t nfb = 0;
    int rc = f.rc;
    if (rc == PMM_OK) rc = pmm_fetch_log10(c, j->out, j->out_capacity, &nfb);
    j->rc = rc; j->n_fallback = nfb;
    if (rc != PMM_OK) j->err = pmm_last_error(c);
}

// Takes the next job off the queue.  wait = false: returns nullptr at once if nothing is queued.  Returns nullptr also
// when the pool is stopping and drained.
static Job* take_job(pmm_pool* p, bool wait)
{
    std::unique_lock<std::mutex> lk(p->mu);
    if (wait) p->cv_work.wait(lk, [&] { return p->stopping || !p->queue.empty(); });
    if (p->queue.empty()) return nullptr;
    Job* j = p->queue.top(); p->queue.pop();
    return j;
}

// A feeder thread drives two contexts of one GPU in turn: it stages and launches a job on one while the job on the other
// is still running, and only then waits for that other one.  So a job is always queued on the GPU behind the one whose
// results the thread is fetching: the host work between two jobs of a context (copy-back, log10, packing the next one,
// about a millisecond) never leaves the GPU idle, and neither does the wake-up of a sleeping wait.  (One thread per
// context -- round 1 -- let all contexts of a GPU fall into step: kernels launched together share the GPU, finish
// together, and the GPU then waits for all their feeders at once; profiles/r02_pool_timeline_n8.jsonl.)
static void feeder_main(pmm_pool* p, size_t slot_a, size_t slot_b)
{
    const size_t slots[2] = {slot_a, slot_b};
    const int n_ctx = slot_b == (size_t)-1 ? 1 : 2;
    Flight fl[2];
    uint64_t seq = 0, started[2] = {0, 0};
    bool stopping = false;
    for (;;) {
        // ---- start a job on every free context: sleep for work only when nothing is in flight; with a job in flight,
        //      take what is waiting or go and deliver that job ---------------------------------------------------------
        for (int k = 0; k < n_ctx && !stopping; ++k) {
            Flight& f = fl[k];
            if (f.active) continue;
            const bool any_active = fl[0].active || fl[1].active;
            if ((f.job = take_job(p, !any_active))) {
                f.t_take = now_s();
                start_job(p->ctxs[slots[k]], f);
                f.active = true; started[k] = ++seq;
            } else if (!any_active) {
                stopping = true;                          // woken with an empty queue: the pool is shutting down
            } else break;
        }
        if (!fl[0].active && !fl[1].active) {
            if (stopping) return;
            continue;
        }
        // ---- finish the older of the jobs in flight ------------------------------------------------------------------------
        const int fin = (fl[0].active && (!fl[1].active || started[0] < started[1])) ? 0 : 1;
        Flight& g = fl[fin];
        {
            pmm_ctx* c = p->ctxs[slots[fin]];
            Job* j = g.job;
            finish_job(c, g);
            const double t_fetched = now_s();
            pmm_pool_trace_t rec{};
            bool have_rec = false;
            if (p->tracing && j->rc == PMM_OK) {          // (read without the lock: a stale value only adds or drops one record)
                pmm_timeline_t tl;
                if (pmm_get_timeline(c, &tl) == PMM_OK) {
                    const double origin = std::chrono::duration<double>(p->t0.time_since_epoch()).count();
                    rec.device = p->ctx_device[slots[fin]]; rec.context = (int32_t)slots[fin];
                    rec.regions = j->num_region; rec.cells = j->cells; rec.pairs = j->pairs;
                    rec.t_take = g.t_take - origin; rec.t_staged = g.t_staged - origin; rec.t_launched = g.t_launched - origin;
                    rec.t_fetched = t_fetched - origin;
                    rec.d_start = tl.ref_host_s + tl.kernels_start_s - origin; rec.d_f32_end = tl.ref_host_s + tl.f32_end_s - origin;
                    rec.d_end = tl.ref_host_s + tl.kernels_end_s - origin;
                    have_rec = true;
                }
            }
            {
                std::lock_guard<std::mutex> lk(p->mu);
                if (have_rec && p->tracing) p->trace.push_back(rec);
                j->device = p->ctx_device[slots[fin]]; j->done = true;
                for (int d = 0; d < p->n_devices; ++d)
                    if (p->devices[d] == j->device) { p->cells_per_device[d] += j->cells; p->jobs_per_device[d]++; }
            }
            p->cv_done.notify_all();
            g.active = false;
        }
    }
}

extern "C" {

int pmm_pool_create(const int* devices, int n_devices, int contexts_per_device, pmm_pool** out)
{
    if (!out) return PMM_ERR_INVALID;
    *out = nullptr;
    const int visible = pmm_device_count();
    if (visible == 0) { g_pool_error = "no CUDA device visible; the pool has no CPU path"; return PMM_ERR_NO_DEVICE; }
    if (contexts_per_device < 1 || contexts_per_device > 8) { g_pool_error = "contexts_per_device must be 1..8"; return PMM_ERR_INVALID; }
    std::vector<int> devs;
    if (!devices || n_devices <= 0) {
        for (int d = 0; d < visible; ++d) devs.push_back(d);        // all GPUs of the box
    } else {
        for (int k = 0; k < n_devices; ++k) {
            if (devices[k] < 0 || devices[k] >= visible) { g_pool_error = "device index out of range"; return PMM_ERR_INVALID; }
            devs.push_back(devices[k]);
        }
    }
    pmm_pool* p = new pmm_pool();
    p->devices = devs; p->n_devices = (int)devs.size();
    p->cells_per_device.assign(devs.size(), 0); p->jobs_per_device.assign(devs.size(), 0);
    for (int rep = 0; rep < contexts_per_device; ++rep)
        for (int d : devs) {
            pmm_ctx* c = nullptr;
            int rc = pmm_create(d, &c);
            if (rc != PMM_OK) {
                g_pool_error = pmm_last_error(nullptr);
                for (pmm_ctx* x : p->ctxs) pmm_destroy(x);
                delete p;
                return rc;
            }
            p->ctxs.push_back(c); p->ctx_device.push_back(d);
        }
    // Waits spin by default.  Measured on an 8-GPU box with 32 host cores (24 feeder threads): spinning 14 100 GCUPS,
    // sleeping on a blocking event 13 400 -- the wake-up latency costs more than the cores it frees.  PMM_POOL_SYNC=block
    // selects the sleeping wait for hosts with fewer cores than feeder threads.
    if (const char* e = getenv("PMM_POOL_SYNC"))
        if (!strcmp(e, "block") || !strcmp(e, "hybrid") || !strcmp(e, "spin") || !strcmp(e, "auto")) for (pmm_ctx* c : p->ctxs) pmm_set_option(c, "sync", e);
    // feeder threads: the contexts of a device in pairs (ctxs is laid out [rep][device])
    const size_t nd = devs.size();
    for (size_t d = 0; d < nd; ++d)
        for (int rep = 0; rep < contexts_per_device; rep += 2) {
            const size_t a = (size_t)rep * nd + d, b = rep + 1 < contexts_per_device ? (size_t)(rep + 1) * nd + d : (size_t)-1;
            p->feeders.emplace_back(feeder_main, p, a, b);
        }
    *out = p;
    return PMM_OK;
}

void pmm_pool_destroy(pmm_pool* p)
{
    if (!p) return;
    {
        std::lock_guard<std::mutex> lk(p->mu);
        p->stopping = true;
    }
    p->cv_work.notify_all();
    for (auto& t : p->feeders) t.join();
    for (pmm_ctx* c : p->ctxs) pmm_destroy(c);
    for (auto& kv : p->jobs) delete kv.second;
    delete p;
}

const char* pmm_pool_last_error(const pmm_pool* p)
{
    if (p) {                                         // a copy taken under the lock: feeders and submitters write p->err
        std::lock_guard<std::mutex> lk(const_cast<pmm_pool*>(p)->mu);
        g_pool_error = p->err;
    }
    return g_pool_error.c_str();
}

int pmm_pool_num_devices(const pmm_pool* p) { return p ? p->n_devices : 0; }

int pmm_pool_submit_flat(pmm_pool* p, uint32_t num_read, const uint32_t* read_off,
                         const uint8_t* bases, const uint8_t* q, const uint8_t* i, const uint8_t* d, const uint8_t* c,
                         uint32_t num_hap, const uint32_t* hap_off, const uint8_t* hap_bases,
                         uint32_t num_region, const pmm_region_t* regions,
                         double* out_log10, uint64_t out_capacity, uint64_t* ticket)
{
    if (!p || !ticket) return PMM_ERR_INVALID;
    if (!read_off || !hap_off || !bases || !q || !i || !d || !c || !hap_bases || !out_log10 || !num_read || !num_hap) {
        std::lock_guard<std::mutex> lk(p->mu);
        p->err = "null or empty input"; return PMM_ERR_INVALID;
    }
    // Validate here, so that a malformed job fails its caller at submit rather than on a feeder, and so that the pool's
    // own reads of it are sound (`cells` below comes from read_off / hap_off at the region bounds): offsets ascend
    // strictly (no read or haplotype of length 0), totals fit.
    {
        const char* bad = nullptr;
        for (uint32_t k = 0; k < num_read && !bad; ++k) if (read_off[k + 1] <= read_off[k]) bad = "read offsets must ascend strictly (no read of length 0)";
        for (uint32_t k = 0; k < num_hap && !bad; ++k) if (hap_off[k + 1] <= hap_off[k]) bad = "haplotype offsets must ascend strictly (no haplotype of length 0)";
        if (!bad && 5ull * (read_off[num_read] - read_off[0]) + (hap_off[num_hap] - hap_off[0]) >= (1ull << 31)) bad = "job larger than 2 GiB: split it";
        if (!bad && regions && num_region)
            for (uint32_t g = 0; g < num_region && !bad; ++g) if (!regions[g].num_read || !regions[g].num_hap) bad = "empty region";
        if (bad) { std::lock_guard<std::mutex> lk(p->mu); p->err = bad; return PMM_ERR_INVALID; }
    }
    Job* j = new Job();
    j->num_read = num_read; j->num_hap = num_hap;
    j->read_off = read_off; j->tr[0] = bases; j->tr[1] = q; j->tr[2] = i; j->tr[3] = d; j->tr[4] = c;
    j->hap_off = hap_off; j->hap = hap_bases;
    if (regions && num_region) { j->regions = regions; j->num_region = num_region; }
    else { j->one_region = pmm_region_t{0, num_read, 0, num_hap}; j->regions = &j->one_region; j->num_region = 1; }
    for (uint32_t g = 0; g < j->num_region; ++g) {
        const pmm_region_t& r = j->regions[g];
        if ((uint64_t)r.read_first + r.num_read > num_read || (uint64_t)r.hap_first + r.num_hap > num_hap) {
            delete j;
            std::lock_guard<std::mutex> lk(p->mu);
            p->err = "region out of range"; return PMM_ERR_INVALID;
        }
        j->pairs += (uint64_t)r.num_read * r.num_hap;
        j->cells += (uint64_t)(read_off[r.read_first + r.num_read] - read_off[r.read_first]) *
                    (uint64_t)(hap_off[r.hap_first + r.num_hap] - hap_off[r.hap_first]);
    }
    if (out_capacity < j->pairs) {
        delete j;
        std::lock_guard<std::mutex> lk(p->mu);
        p->err = "output buffer too small"; return PMM_ERR_INVALID;
    }
    j->out = out_log10; j->out_capacity = out_capacity;
    {
        std::lock_guard<std::mutex> lk(p->mu);
        if (p->stopping) { delete j; p->err = "pool is shutting down"; return PMM_ERR_STATE; }
        j->ticket = p->next_ticket++;
        j->generation = j->ticket / (2 * p->ctxs.size() + 1);      // about two jobs per context
        p->jobs[j->ticket] = j;
        p->queue.push(j);
        *ticket = j->ticket;
    }
    p->cv_work.notify_one();
    return PMM_OK;
}

int pmm_pool_wait(pmm_pool* p, uint64_t ticket, uint64_t* n_fallback, int* device)
{
    if (!p) return PMM_ERR_INVALID;
    std::unique_lock<std::mutex> lk(p->mu);
    auto it = p->jobs.find(ticket);
    if (it == p->jobs.end()) { p->err = "unknown ticket"; return PMM_ERR_STATE; }
    Job* j = it->second;
    p->cv_done.wait(lk, [&] { return j->done; });
    const int rc = j->rc;
    if (rc != PMM_OK) p->err = j->err;
    if (n_fallback) *n_fallback = j->n_fallback;
    if (device) *device = j->device;
    p->jobs.erase(it);
    delete j;
    return rc;
}

int pmm_pool_trace(pmm_pool* p, int on)
{
    if (!p) return PMM_ERR_INVALID;
    std::lock_guard<std::mutex> lk(p->mu);
    if (on) p->trace.clear();
    p->tracing = on != 0;
    return PMM_OK;
}

int pmm_pool_get_trace(pmm_pool* p, pmm_pool_trace_t* out, uint64_t capacity, uint64_t* count)
{
    if (!p || !count) return PMM_ERR_INVALID;
    std::lock_guard<std::mutex> lk(p->mu);
    *count = p->trace.size();
    if (out) memcpy(out, p->trace.data(), sizeof(pmm_pool_trace_t) * std::min<uint64_t>(capacity, p->trace.size()));
    return PMM_OK;
}

int pmm_pool_device_load(const pmm_pool* p, int slot, int* device, uint64_t* jobs, uint64_t* cells)
{
    if (!p || slot < 0 || slot >= p->n_devices) return PMM_ERR_INVALID;
    std::lock_guard<std::mutex> lk(const_cast<pmm_pool*>(p)->mu);
    if (device) *device = p->devices[slot];
    if (jobs) *jobs = p->jobs_per_device[slot];
    if (cells) *cells = p->cells_per_device[slot];
    return PMM_OK;
}

}  // extern "C"
