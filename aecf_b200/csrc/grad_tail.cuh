// Host-side interface of the backward's gradient tail (grad_tail.cu) and of the cross-rank sum it can contain
// (peer_allreduce.cu).
#pragma once

#include "gemm.cuh"

namespace aecf {

// Offsets (in floats, all multiples of 4) of the raw gradient sums S of the folded backward.
struct TailLayout { long long g, o, bo, pool, total; };
inline TailLayout tail_layout(int D, int HSP) {
    TailLayout t;
    t.g = 0;                                                    // [dWv ; R]              (D + HSP) x D
    t.o = t.g + static_cast<long long>(D + HSP) * D;            // dWo                    D x D
    t.bo = t.o + static_cast<long long>(D) * D;                 // colsum(d_out)          D
    t.pool = t.bo + D;                                          // pool bias sums         3 D: [d_q | d_bias_v | d_bias_k]
    t.total = (t.pool + 3LL * D + 3) & ~3LL;
    return t;
}

struct GradTailArgs {
    int dtype, D, H, HSP, sms;
    int grad_dtype;                     // of d_in_w ... d_query: dtype, or fp32 next to bf16 parameters (mixed precision)
    GemmPartials g, o;                  // [dWv ; R] and dWo as left by gemm_partials (o.partial null: no dWo wanted)
    const void* d_out; long long rows;  // column sums of d_out -> d_out_proj_bias (null: not wanted)
    // the pool backward's per-sample [s | sum_m ds] ([samples][2 HSP] fp32) and d_ctx: d_bias_v = sum_b s[b, h] d_ctx[b, :],
    // d_bias_k = scale q sum_b sum_m ds (null: in_proj_bias gradient not wanted)
    const float* rowsum; const void* d_ctx; long long samples;
    // ... or, when the weights of every sample sum to one: d_bias_v = Wo^T colsum(d_out), d_bias_k = 0 (null: not this way)
    const void* out_proj_weight;
    float* sums;                        // S, tail_layout(D, HSP).total floats
    void* scratch;                      // grad_tail_scratch_bytes(D, sms)
    const float* q_proj; const void* in_proj_weight; const void* query;
    void *d_in_w, *d_in_b, *d_out_w, *d_out_b, *d_query;
};

size_t grad_tail_scratch_bytes(int D, int sms);
enum { GATHER_EARLY = 0, GATHER_LATE = 1 };
int launch_grad_gather(const GradTailArgs& a, int which, cudaStream_t s);
int launch_grad_finish(const GradTailArgs& a, const float* sums, cudaStream_t s);
// peer_allreduce.cu: dst[r][i] = (1/world if average) * sum_r' src[r'][i] for every rank r, fp32, `count` floats
int launch_peer_sum(int device, const aecf_dp_desc* dp, long long count, cudaStream_t s);

}  // namespace aecf
