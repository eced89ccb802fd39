// host_workers.cpp -- see host_workers.h.
#include "host_workers.h"

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <mutex>
#include <thread>
#include <vector>

namespace {

// Host worker threads for the per-result log10 (the one piece of the path that stays on the host so that it uses the
// host libm like the reference).  Created once per process on first use; a fetch hands out chunks and takes part
// itself, so small jobs never wait for a wake-up.  A call that finds the workers taken runs on its own thread.
class HostWorkers {
 public:
    static HostWorkers& get() { static HostWorkers w; return w; }
    void run(uint64_t n, uint64_t grain, const std::function<void(uint64_t, uint64_t)>& f)
    {
        if (n <= grain || th_.empty()) { f(0, n); return; }
        // Workers busy with another context's results: the process is streaming jobs through several contexts, and
        // the caller's own thread is the parallelism (24 feeder threads on an 8-GPU box) -- do not queue up behind them.
        std::unique_lock<std::mutex> call(call_mu_, std::try_to_lock);
        if (!call.owns_lock()) { f(0, n); return; }
        {
            std::lock_guard<std::mutex> lk(mu_);
            fn_ = &f; n_ = n; grain_ = grain; next_.store(0); busy_ = (int)th_.size(); ++gen_;
        }
        cv_work_.notify_all();
        work();
        std::unique_lock<std::mutex> lk(mu_);
        cv_done_.wait(lk, [&] { return busy_ == 0; });
        fn_ = nullptr;
    }

 private:
    HostWorkers()
    {
        const unsigned hw = std::thread::hardware_concurrency();
        const unsigned n = hw > 1 ? std::min(hw - 1, 7u) : 0;
        for (unsigned k = 0; k < n; ++k) th_.emplace_back([this] { loop(); });
    }
    ~HostWorkers()
    {
        { std::lock_guard<std::mutex> lk(mu_); stop_ = true; }
        cv_work_.notify_all();
        for (auto& t : th_) t.join();
    }
    void work()
    {
        for (;;) {
            const uint64_t a = next_.fetch_add(grain_);
            if (a >= n_) return;
            (*fn_)(a, std::min(n_, a + grain_));
        }
    }
    void loop()
    {
        uint64_t seen = 0;
        for (;;) {
            {
                std::unique_lock<std::mutex> lk(mu_);
                cv_work_.wait(lk, [&] { return stop_ || gen_ != seen; });
                if (stop_) return;
                seen = gen_;
            }
            work();
            { std::lock_guard<std::mutex> lk(mu_); --busy_; }
            cv_done_.notify_one();
        }
    }
    std::vector<std::thread> th_;
    std::mutex mu_, call_mu_;
    std::condition_variable cv_work_, cv_done_;
    const std::function<void(uint64_t, uint64_t)>* fn_ = nullptr;
    uint64_t n_ = 0, grain_ = 1, gen_ = 0;
    std::atomic<uint64_t> next_{0};
    int busy_ = 0;
    bool stop_ = false;
};

}  // namespace

namespace pmm {

void host_parallel_for(uint64_t n, uint64_t grain, const std::function<void(uint64_t, uint64_t)>& f)
{
    HostWorkers::get().run(n, std::max<uint64_t>(grain, 1), f);
}

}  // namespace pmm
