// sw_engine.cu -- the C ABI of include/smithwaterman_cuda.h: validation, chunking by backtrack-memory budget, largest
// pairs first, one kernel launch per chunk, results back.  Stands where the reference has its per-pair CPU loop
// (/root/reference/htc-sw/host/FalconSW_AVX.cpp:304-313) and the FPGA dispatch (host/sw_host.cpp:13-15).  No CPU path.
#include "../../include/smithwaterman_cuda.h"
#include "cuda_util.h"
#include "host_workers.h"
#include "sw_kernels.cuh"

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <string>
#include <vector>

using namespace sw;

namespace {
std::string g_sw_create_error;
}  // namespace

constexpr uint64_t kCigarScratchBytes = 256ull << 20;   // per-chunk scratch rows of the traceback (cigar_cap elements per pair)

struct sw_ctx {
    int device = 0, sm_count = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[2] = {nullptr, nullptr};
    std::string err;
    DevBuf d_seq1, d_seq2, d_pairs, d_bt, d_cigars, d_compact, d_first, d_nelem, d_off, d_score, d_counter;
    PinBuf h_stage, h_out, h_cig;
    uint64_t compact_hint = 16;                   // CIGAR elements per pair the compact array is sized for (grows on overflow)
    uint64_t bt_budget_words = (1ull << 30);      // 4 GiB of backtrack codes per chunk
    sw_stats_t stats{};
    int fail(int code, const std::string& m) { err = m; return code; }
    int fail_cuda(cudaError_t e, const char* what) { err = std::string(what) + ": " + cudaGetErrorString(e); return SW_ERR_CUDA; }
};

#define SW_CUDA(ctx, call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return (ctx)->fail_cuda(e__, #call); } while (0)

extern "C" {

int sw_create(int device, sw_ctx** out)
{
    if (!out) return SW_ERR_INVALID;
    *out = nullptr;
    int sm_count = 0;
    const int rc = open_device<SW_ERR_INVALID, SW_ERR_CUDA, SW_ERR_NO_DEVICE>(device, sm_count, g_sw_create_error, "the aligner");
    if (rc) return rc;
    sw_ctx* c = new sw_ctx();
    c->device = device; c->sm_count = sm_count;
    const cudaError_t e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) { g_sw_create_error = cudaGetErrorString(e); delete c; return SW_ERR_CUDA; }
    cudaEventCreate(&c->ev[0]); cudaEventCreate(&c->ev[1]);
    *out = c;
    return SW_OK;
}

void sw_destroy(sw_ctx* c)
{
    if (!c) return;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    cudaEventDestroy(c->ev[0]); cudaEventDestroy(c->ev[1]);
    cudaStreamDestroy(c->stream);
    delete c;
}

const char* sw_last_error(const sw_ctx* c) { return c ? c->err.c_str() : g_sw_create_error.c_str(); }

int sw_get_stats(const sw_ctx* c, sw_stats_t* out)
{
    if (!c || !out) return SW_ERR_INVALID;
    *out = c->stats;
    return SW_OK;
}

int sw_align_batch(sw_ctx* c, uint32_t n_pairs,
                   const uint8_t* seq1_bytes, const uint32_t* seq1_start, const uint32_t* seq1_len,
                   const uint8_t* seq2_bytes, const uint32_t* seq2_start, const uint32_t* seq2_len,
                   int w_match, int w_mismatch, int w_open, int w_extend, int overhang_strategy,
                   uint32_t cigar_cap, sw_cigar_elem_t* cigars, int32_t* n_elem, int32_t* alignment_offset, int32_t* score)
{
    if (!c) return SW_ERR_INVALID;
    if (!n_pairs) return SW_OK;
    if (!seq1_bytes || !seq1_start || !seq1_len || !seq2_bytes || !seq2_start || !seq2_len || !cigars || !n_elem || !alignment_offset)
        return c->fail(SW_ERR_INVALID, "null argument");
    if (overhang_strategy < 0 || overhang_strategy > 3) return c->fail(SW_ERR_INVALID, "unknown overhang strategy");
    if (!cigar_cap) return c->fail(SW_ERR_INVALID, "cigar_cap must be positive");
    // within this domain no score or tie-break difference of the fill can overflow (see cells() in sw_kernels.cu)
    for (const int w : {w_match, w_mismatch, w_open, w_extend})
        if (w < -kMaxWeight || w > kMaxWeight) return c->fail(SW_ERR_INVALID, "weight outside [-65536, 65536]");
    const auto t0 = std::chrono::steady_clock::now();
    static const bool trace = getenv("SW_TRACE") != nullptr;
    auto mark = [&](const char* what) { if (trace) fprintf(stderr, "[sw] %-10s %.3f ms\n", what, std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count()); };
    cudaSetDevice(c->device);
    cudaStream_t s = c->stream;

    uint64_t ext1 = 0, ext2 = 0, cells = 0;
    for (uint32_t p = 0; p < n_pairs; ++p) {
        if (!seq1_len[p] || !seq2_len[p]) return c->fail(SW_ERR_INVALID, "sequence of length 0");
        if (seq1_len[p] > (uint32_t)kMaxLen || seq2_len[p] > (uint32_t)kMaxLen) return c->fail(SW_ERR_INVALID, "sequence longer than 4095 bases");
        ext1 = std::max<uint64_t>(ext1, (uint64_t)seq1_start[p] + seq1_len[p]);
        ext2 = std::max<uint64_t>(ext2, (uint64_t)seq2_start[p] + seq2_len[p]);
        cells += (uint64_t)seq1_len[p] * seq2_len[p];
    }
    if (ext1 >= (1ull << 31) || ext2 >= (1ull << 31)) return c->fail(SW_ERR_INVALID, "sequence blobs larger than 2 GiB");

    // largest pairs first: warps pull pairs in order, the tail of the launch is made of the small ones.  A stable
    // counting sort on 4096 size classes (cells / 4096), linear in the number of pairs: the order inside a class does
    // not matter for the tail.
    std::vector<uint32_t> order(n_pairs);
    {
        constexpr uint32_t kClasses = 4096;                              // cells < 2^24
        std::vector<uint32_t> first(kClasses + 1, 0);
        auto cls = [&](uint32_t p) { return kClasses - 1 - (uint32_t)(((uint64_t)seq1_len[p] * seq2_len[p]) >> 12); };
        for (uint32_t p = 0; p < n_pairs; ++p) ++first[cls(p) + 1];
        for (uint32_t k = 0; k < kClasses; ++k) first[k + 1] += first[k];
        for (uint32_t p = 0; p < n_pairs; ++p) order[first[cls(p)]++] = p;
    }

    mark("sorted");
    SW_CUDA(c, c->d_seq1.reserve(ext1)); SW_CUDA(c, c->d_seq2.reserve(ext2));
    SW_CUDA(c, c->h_stage.reserve(ext1 + ext2 + sizeof(PairDesc) * (size_t)n_pairs + 64));
    SW_CUDA(c, c->d_pairs.reserve(sizeof(PairDesc) * (size_t)n_pairs));
    // CIGARs are a few elements per pair, not cigar_cap of them (callers pass the longest sequence, ~12 KB per pair): the
    // compact array is sized from an estimate and the batch repeated with more room if it ever runs over; the per-pair
    // scratch rows exist per chunk, not per batch (see the chunk loop)
    const uint64_t compact_cap = std::min<uint64_t>((uint64_t)n_pairs * cigar_cap, std::max<uint64_t>((uint64_t)n_pairs * c->compact_hint, 1u << 16));
    SW_CUDA(c, c->d_compact.reserve(sizeof(int2) * compact_cap));
    SW_CUDA(c, c->d_first.reserve(sizeof(uint32_t) * (size_t)n_pairs));
    SW_CUDA(c, c->d_nelem.reserve(sizeof(int32_t) * (size_t)n_pairs));
    SW_CUDA(c, c->d_off.reserve(sizeof(int32_t) * (size_t)n_pairs));
    SW_CUDA(c, c->d_score.reserve(sizeof(int32_t) * (size_t)n_pairs));
    SW_CUDA(c, c->d_counter.reserve(256));
    char* hs = static_cast<char*>(c->h_stage.p);
    auto copy_in = [&](char* dst, const uint8_t* src, uint64_t n) {       // into pinned memory, by the host workers
        pmm::host_parallel_for(n, 1 << 18, [&](uint64_t b0, uint64_t b1) { memcpy(dst + b0, src + b0, b1 - b0); });
    };
    copy_in(hs, seq1_bytes, ext1); copy_in(hs + ext1, seq2_bytes, ext2);
    SW_CUDA(c, cudaMemcpyAsync(c->d_seq1.p, hs, ext1, cudaMemcpyHostToDevice, s));
    SW_CUDA(c, cudaMemcpyAsync(c->d_seq2.p, hs + ext1, ext2, cudaMemcpyHostToDevice, s));

    // chunks: consecutive pairs (in size order) whose backtrack matrices fit the budget
    PairDesc* hp = reinterpret_cast<PairDesc*>(hs + ((ext1 + ext2 + 15) & ~(size_t)15));
    std::vector<std::pair<uint32_t, uint32_t>> chunks;     // [first, last) in `order`
    uint64_t max_words = 0;
    for (uint32_t k = 0; k < n_pairs;) {
        uint64_t words = 0; const uint32_t first = k;
        while (k < n_pairs) {
            const uint32_t p = order[k];
            const uint32_t stride = (seq2_len[p] + 31 + 7) / 8;      // words per row: codes are indexed by step (l2 + 31 of them)
            // blocks of 32 x K rows, every block [word][lane][row of the lane]: rows are padded to whole blocks
            const uint32_t K = pick_rows_per_lane(seq1_len[p]);
            const uint64_t w = (uint64_t)((seq1_len[p] + 32 * K - 1) / (32 * K)) * 32 * K * stride;
            if (k > first && (words + w > c->bt_budget_words || (uint64_t)(k - first + 1) * cigar_cap * sizeof(int2) > kCigarScratchBytes)) break;
            hp[k] = PairDesc{seq1_start[p], seq1_len[p], seq2_start[p], seq2_len[p], words, stride, p, K, 0u};
            words += w; ++k;
        }
        chunks.emplace_back(first, k);
        max_words = std::max(max_words, words);
    }
    SW_CUDA(c, c->d_bt.reserve(max_words * sizeof(uint32_t)));
    {
        uint64_t most = 1;
        for (const auto& ch : chunks) most = std::max<uint64_t>(most, ch.second - ch.first);
        SW_CUDA(c, c->d_cigars.reserve(sizeof(int2) * most * cigar_cap));
    }
    SW_CUDA(c, cudaMemcpyAsync(c->d_pairs.p, hp, sizeof(PairDesc) * (size_t)n_pairs, cudaMemcpyHostToDevice, s));

    mark("staged");
    uint32_t launches = 0;
    uint32_t* d_count = static_cast<uint32_t*>(c->d_counter.p) + 32;      // compact CIGAR cursor, its own 128-byte line
    SW_CUDA(c, cudaMemsetAsync(d_count, 0, sizeof(uint32_t), s));
    SW_CUDA(c, cudaEventRecord(c->ev[0], s));
    for (const auto& ch : chunks) {
        Args a{};
        a.seq1 = static_cast<uint8_t*>(c->d_seq1.p); a.seq2 = static_cast<uint8_t*>(c->d_seq2.p);
        a.pairs = static_cast<PairDesc*>(c->d_pairs.p) + ch.first; a.npairs = ch.second - ch.first;
        a.counter = static_cast<uint32_t*>(c->d_counter.p);
        a.bt = static_cast<uint32_t*>(c->d_bt.p);
        a.match = w_match; a.mismatch = w_mismatch; a.open = w_open; a.extend = w_extend; a.strategy = overhang_strategy;
        a.cigar_cap = cigar_cap; a.cigars = static_cast<int2*>(c->d_cigars.p);
        a.compact = static_cast<int2*>(c->d_compact.p); a.compact_cap = (uint32_t)std::min<uint64_t>(compact_cap, 0xffffffffu); a.compact_count = d_count; a.compact_first = static_cast<uint32_t*>(c->d_first.p);
        a.n_elem = static_cast<int32_t*>(c->d_nelem.p); a.offset = static_cast<int32_t*>(c->d_off.p);
        a.score = static_cast<int32_t*>(c->d_score.p);
        a.max_l1 = 0; a.max_l2 = 0;
        a.k_neg1 = -1; a.k_one = 1;
        for (uint32_t k = ch.first; k < ch.second; ++k) { a.max_l1 = std::max(a.max_l1, hp[k].l1); a.max_l2 = std::max(a.max_l2, hp[k].l2); }
        SW_CUDA(c, cudaMemsetAsync(a.counter, 0, sizeof(uint32_t), s));
        SW_CUDA(c, launch_align(a, c->sm_count, s, nullptr));
        ++launches;
    }
    SW_CUDA(c, cudaEventRecord(c->ev[1], s));

    mark("launched");
    // Results: the per-pair integers and the number of CIGAR elements first, then the compact CIGAR array (a few
    // elements per pair, contiguous) which is scattered into the caller's rows of cigar_cap elements here.
    const size_t sz_i = sizeof(int32_t) * (size_t)n_pairs;
    SW_CUDA(c, c->h_out.reserve(4 * sz_i + 64));
    char* ho = static_cast<char*>(c->h_out.p);
    SW_CUDA(c, cudaMemcpyAsync(ho, c->d_nelem.p, sz_i, cudaMemcpyDeviceToHost, s));
    SW_CUDA(c, cudaMemcpyAsync(ho + sz_i, c->d_off.p, sz_i, cudaMemcpyDeviceToHost, s));
    SW_CUDA(c, cudaMemcpyAsync(ho + 2 * sz_i, c->d_score.p, sz_i, cudaMemcpyDeviceToHost, s));
    SW_CUDA(c, cudaMemcpyAsync(ho + 3 * sz_i, c->d_first.p, sz_i, cudaMemcpyDeviceToHost, s));
    SW_CUDA(c, cudaMemcpyAsync(ho + 4 * sz_i, d_count, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    SW_CUDA(c, cudaStreamSynchronize(s));
    mark("synced");
    memcpy(n_elem, ho, sz_i);
    memcpy(alignment_offset, ho + sz_i, sz_i);
    if (score) memcpy(score, ho + 2 * sz_i, sz_i);
    static_assert(sizeof(sw_cigar_elem_t) == sizeof(int2), "cigar element layout");
    uint32_t total = 0;
    memcpy(&total, ho + 4 * sz_i, sizeof total);
    if (total > compact_cap) {
        // more CIGAR elements than the estimate allowed for: remember, and run the batch again with room for all of them
        c->compact_hint = std::max<uint64_t>(c->compact_hint * 2, ((uint64_t)total + n_pairs - 1) / n_pairs + 1);
        return sw_align_batch(c, n_pairs, seq1_bytes, seq1_start, seq1_len, seq2_bytes, seq2_start, seq2_len, w_match, w_mismatch,
                              w_open, w_extend, overhang_strategy, cigar_cap, cigars, n_elem, alignment_offset, score);
    }
    if (total) {
        SW_CUDA(c, c->h_cig.reserve(sizeof(int2) * (size_t)total));
        const int2* hc = static_cast<const int2*>(c->h_cig.p);
        SW_CUDA(c, cudaMemcpyAsync(const_cast<int2*>(hc), c->d_compact.p, sizeof(int2) * (size_t)total, cudaMemcpyDeviceToHost, s));
        SW_CUDA(c, cudaStreamSynchronize(s));
        const uint32_t* first = reinterpret_cast<const uint32_t*>(ho + 3 * sz_i);
        pmm::host_parallel_for(n_pairs, 1024, [&](uint64_t p0, uint64_t p1) {
            for (uint64_t p = p0; p < p1; ++p) {
                const uint32_t stored = std::min<uint32_t>(cigar_cap, (uint32_t)std::max(0, n_elem[p]));
                memcpy(cigars + (size_t)p * cigar_cap, hc + first[p], sizeof(int2) * (size_t)stored);
            }
        });
    }

    mark("scattered");
    c->stats = sw_stats_t{};
    c->stats.pairs = n_pairs; c->stats.cells = cells; c->stats.bytes_backtrack = max_words * sizeof(uint32_t);
    c->stats.kernel_launches = launches; c->stats.chunks = (uint32_t)chunks.size();
    cudaEventElapsedTime(&c->stats.ms_kernel, c->ev[0], c->ev[1]);
    c->stats.ms_total = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    return SW_OK;
}

}  // extern "C"
