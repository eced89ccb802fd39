// host_workers.h -- the library's host worker threads (host_workers.cpp), shared by both engines: the PairHMM fetch
// takes log10 on them, the Smith-Waterman path stages and scatters CIGARs on them.
#pragma once
#include <cstdint>
#include <functional>

namespace pmm {

// Runs f(a, b) over [0, n) in chunks of `grain`, on the workers and the calling thread.
void host_parallel_for(uint64_t n, uint64_t grain, const std::function<void(uint64_t, uint64_t)>& f);

}  // namespace pmm
