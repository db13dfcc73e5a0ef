// Optional per-kernel timing: CUDA events recorded immediately around each launch, on the launching stream.
#include <cstdio>
#include <mutex>
#include <vector>

#include "common.cuh"

namespace aecf {

namespace {
struct Record { int site; cudaEvent_t a, b; };
struct Timing {
    std::mutex mu;
    bool on = false;
    std::vector<Record> records;
    std::vector<cudaEvent_t> pool;            // events are created once and reused
    size_t pool_used = 0;
    cudaEvent_t take() {
        if (pool_used == pool.size()) {
            cudaEvent_t e;
            if (cudaEventCreate(&e) != cudaSuccess) return nullptr;
            pool.push_back(e);
        }
        return pool[pool_used++];
    }
};
Timing g_timing;
thread_local int g_site = AECF_SITE_OTHER;
const char* kSiteNames[AECF_SITE_COUNT] = {
    "other", "q_proj", "kv_proj", "pool_fwd", "out_proj", "d_out_bias", "d_out_weight", "d_ctx", "pool_bwd",
    "pool_bwd_finalize", "d_x", "d_kv_weight", "d_q_weight", "d_query", "d_in_bias", "entropy_loss", "fold_prepare",
    "fold_finish", "grad_gather", "grad_peer_sum", "grad_finish", "param_cast"};
char g_site_gemm[AECF_SITE_COUNT][96];                 // the GEMM kernel last launched from each site (diagnostics)
}  // namespace

void note_site_gemm_kernel(const char* name) {
    std::lock_guard<std::mutex> lock(g_timing.mu);
    std::snprintf(g_site_gemm[g_site], sizeof(g_site_gemm[0]), "%s", name);
}

ScopedSite::ScopedSite(int site) : previous(g_site) { g_site = site; }
ScopedSite::~ScopedSite() { g_site = previous; }

int timing_begin(cudaStream_t s, int site_override) {
    if (!g_timing.on) return -1;
    std::lock_guard<std::mutex> lock(g_timing.mu);
    if (!g_timing.on) return -1;
    Record r;
    r.site = site_override >= 0 ? site_override : g_site;
    r.a = g_timing.take();
    r.b = g_timing.take();
    if (!r.a || !r.b) return -1;
    cudaEventRecord(r.a, s);
    g_timing.records.push_back(r);
    return static_cast<int>(g_timing.records.size()) - 1;
}

void timing_end(int record, cudaStream_t s) {
    std::lock_guard<std::mutex> lock(g_timing.mu);
    if (record >= 0 && record < static_cast<int>(g_timing.records.size())) cudaEventRecord(g_timing.records[record].b, s);
}

}  // namespace aecf

using namespace aecf;

extern "C" {

int aecf_timing_enable(int32_t enable) {
    std::lock_guard<std::mutex> lock(g_timing.mu);
    g_timing.on = enable != 0;
    g_timing.records.clear();
    g_timing.pool_used = 0;
    return AECF_OK;
}

int aecf_timing_collect(float* total_ms, int32_t* launches) {
    if (!total_ms || !launches) return AECF_ERR_INVALID;
    std::lock_guard<std::mutex> lock(g_timing.mu);
    for (int i = 0; i < AECF_SITE_COUNT; ++i) { total_ms[i] = 0.f; launches[i] = 0; }
    for (const Record& r : g_timing.records) {
        AECF_CUDA_OK(cudaEventSynchronize(r.b));
        float ms = 0.f;
        AECF_CUDA_OK(cudaEventElapsedTime(&ms, r.a, r.b));
        total_ms[r.site] += ms;
        launches[r.site] += 1;
    }
    g_timing.records.clear();
    g_timing.pool_used = 0;
    return AECF_OK;
}

const char* aecf_timing_site_gemm_kernel(int32_t site) {
    return (site >= 0 && site < AECF_SITE_COUNT) ? g_site_gemm[site] : "";
}

const char* aecf_timing_site_name(int32_t site) {
    return (site >= 0 && site < AECF_SITE_COUNT) ? kSiteNames[site] : "invalid";
}

}  // extern "C"
