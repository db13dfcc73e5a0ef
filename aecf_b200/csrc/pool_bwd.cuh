// Fused pool backward (recompute), persistent over rows.
//
// Re-derives the softmax/dropout weights from q and kv (nothing is saved by the forward: this is
// the recompute the reference's use_checkpoint= flag asks torch.utils.checkpoint for, reference
// aecf/AECFLayer.py:501-512), then emits dK and dV straight into the packed d_kv buffer and
// accumulates the three batch reductions that share its data:
//     d_q (shared query)  = scale * sum_b sum_m ds[b,h,m] k[b,m,h,:]
//     d_bias_v            = sum_b,m dV      d_bias_k = sum_b,m dK   (analytically ~0)
// Closed form: SURVEY.md Appendix B; the autograd graph it replaces is that of
// torch/nn/functional.py:6632-6647, 6657-6659.
// HBM-bound: algorithmic bytes per sample = s*(2*M*D + D + 2*M*D)  (SURVEY.md section 8d).
//
// The batch sums live in shared memory (one private strip per warp, lane-contiguous float4 so
// the read-modify-write is conflict free), not in registers: that keeps the kernel at two CTAs
// per SM.  They are folded in a fixed order at the end, so results are run-to-run identical.
#pragma once

#include "pool_core.cuh"

namespace aecf {

template <int J, int V>
struct BwdSmem {
    static constexpr int ACC = J * V * 32;               // floats per accumulator strip
    static constexpr int PER_WARP = 2 * ACC + J * 32;    // acc_q | acc_bv | acc_sds
    static constexpr int bytes(int M) { return (POOL_WARPS * M + POOL_WARPS * PER_WARP) * 4; }
};

// strip[j][.][lane] += a * x: one of a warp's batch-sum strips ([J][V / 4][32] float4).  The head-mean gradient, the
// softmax backward and the strip fold are also in pool_bwd_multi_kernel, but stay inline in both: as shared helpers
// they changed the SASS of 134, 365 and 328 of the 768 backward kernels (scripts/sass_diff.py).
template <int V>
__device__ __forceinline__ void strip_fma(float4* strip, int j, int lane, float a, const float (&x)[V]) {
    constexpr int Q4 = V / 4;
#pragma unroll
    for (int q4 = 0; q4 < Q4; ++q4) {
        float4 t = strip[(j * Q4 + q4) * 32 + lane];
        t.x = fmaf(a, x[4 * q4], t.x); t.y = fmaf(a, x[4 * q4 + 1], t.y);
        t.z = fmaf(a, x[4 * q4 + 2], t.z); t.w = fmaf(a, x[4 * q4 + 3], t.w);
        strip[(j * Q4 + q4) * 32 + lane] = t;
    }
}

// FOLD (folded key projection, DESIGN.md): kv holds the values only, the scores come precomputed, there is no
// key pass -- the score gradient ds[b, m, h] itself is stored next to dV (d_kv rows are [dV (D) | ds (HSP)]) and
// the dX / dW GEMMs that follow contract over D + HSP, which applies and accumulates the rank-H key-side terms.
// PAD: the padded lane map (pool_core.cuh).
template <typename T, int M, int J, bool DROP, bool FOLD, bool PAD>
// The folded variant has no key pass and fits 80 registers without spilling for M * J <= 10 (ptxas -v): three CTAs
// per SM instead of two, i.e. half as many loads again in flight for a kernel that waits on HBM latency
// (ncu r1 run 18: long-scoreboard stalls dominate, 25 % of the warp slots occupied).
__global__ void __launch_bounds__(POOL_WARPS * 32, (FOLD && M * J <= 10 && J <= 2) ? 3 : 2)
pool_bwd_kernel(const PoolParams p) {
    using Core = PoolCore<T, M, J, DROP, PAD>;
    using Smem = BwdSmem<J, Core::V>;
    constexpr int V = Core::V;
    constexpr int Q4 = V / 4;
    constexpr int VHALF = FOLD ? 0 : 1;
    // Every load of a row -- d_ctx, K and (when it fits in registers) V -- is issued before any
    // arithmetic, so a warp makes one trip to HBM per row.  K is needed again for d_q after the softmax
    // backward; it is re-read through L1 (the first read allocates there) rather than held in registers.
    constexpr bool PRELOAD_V = (M * J <= 8);

    AECF_DYNAMIC_SMEM_ALIGNED16(float, smem);
    float* xchg = smem;                                               // [POOL_WARPS][M]
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    float* strip = smem + POOL_WARPS * M + warp * Smem::PER_WARP;     // this warp's accumulators
    float4* acc_q = reinterpret_cast<float4*>(strip);                 // [J][Q4][32]
    float4* acc_bv = reinterpret_cast<float4*>(strip + Smem::ACC);    // [J][Q4][32]
    float* acc_sds = strip + 2 * Smem::ACC;                           // [J][32]
    // Folded backward inside aecf_fusion_bwd (p.partials == null): no batch sums here at all.  Without cross-sample state a
    // CTA costs nothing to start or to retire, which is what makes the chunked schedule below pay (r2 run 20: 86.3 us
    // persistent, 80.3 us in chunks of 32; with a per-CTA fold of the strips the chunks LOSE 8 us).  The sums in question
    // are the value and key thirds of the in-projection bias gradient:
    //   d_bias_v[d] = sum_b s[b, h(d)] d_ctx[b, d],  s = sum_m wd       d_bias_k[d] = scale q[d] sum_b sum_m ds[b, m, h(d)]
    // Without dropout s = sum_m softmax = 1 and sum_m ds = 0 identically, so d_bias_v = sum_b d_ctx[b, :] = Wo^T d_bias_o and
    // d_bias_k = 0: the gradient tail forms them from the column sums of d_out it already has (grad_tail.cu), and nothing is
    // left to do here (p.rowsum == null).  With dropout, a mask, or when only listed samples are pooled, the kernel leaves
    // [s | sum_m ds] per sample and head in p.rowsum and the tail walks d_ctx once more.
    const bool sums = p.partials != nullptr;
    if (sums) for (int i = lane; i < Smem::PER_WARP; i += 32) strip[i] = 0.f;
    __syncwarp();
    pdl_wait();
    const RngKey rng = effective_rng(p.rng, p.rng_state);

    const int slice = warp % p.WPS;
    const int c0 = slice * Core::CPW + lane;

    float qs[J][V];
    if (!FOLD && p.q_shared) Core::load_query(p, 0, c0, qs);

    // Two schedules.  chunk == 0: persistent, CTAs stride over the batch.  chunk > 0: CTA b owns the `chunk` consecutive
    // samples from b * chunk and the grid is as long as the batch needs -- the hardware's block scheduler hands the chunks
    // out as CTAs retire, which evens out the SMs' unequal shares of the memory system (r2 runs 15-17: the bare memory
    // skeleton of this kernel runs 81.7 us persistent and 77.5 / 75.9 / 74.3 us with 32 / 16 / 8 samples per CTA).
    // Either way a CTA's partial sums cover a set of samples that depends on the launch geometry only: bit-reproducible.
    const long long stride = p.chunk ? p.SPC : static_cast<long long>(gridDim.x) * p.SPC;
    const long long first = p.chunk ? static_cast<long long>(blockIdx.x) * p.chunk : static_cast<long long>(blockIdx.x) * p.SPC;
    const long long last = p.chunk ? min(p.B, first + p.chunk) : p.B;
    for (long long base = first; base < last; base += stride) {
        const long long row_raw = base + warp / p.WPS;
        const bool row_ok = row_raw < last;
        const long long row = row_ok ? row_raw : p.B - 1;
        if (!FOLD && !p.q_shared) Core::load_query(p, row, c0, qs);
        const long long src = source_row(p, row);          // where the row's sample lives in kv / scores / d_ctx / d_kv

        const char* kv_row = static_cast<const char*>(p.kv) + Core::row_offset(p, src, c0);
        char* dkv_row = static_cast<char*>(p.d_kv) + Core::drow_offset(p, src, c0);
        auto valid = [&](int j) { return Core::valid(p, c0, j); };

        // upstream gradient of the context and the values, issued first
        uint4 dcraw[J];
        Core::load_row(p, p.d_ctx, src, c0, dcraw);
        uint4 vraw[PRELOAD_V ? M : 1][PRELOAD_V ? J : 1];
        if (PRELOAD_V) {
#pragma unroll
            for (int m = 0; m < M; ++m)
#pragma unroll
                for (int j = 0; j < J; ++j)
                    vraw[PRELOAD_V ? m : 0][PRELOAD_V ? j : 0] =
                        valid(j) ? ldg_stream(kv_row + Core::kv_rel(p, c0, m, VHALF, j)) : make_uint4(0, 0, 0, 0);
        }

        float w[M][J], wd[M][J];
        unsigned keep;
        if constexpr (FOLD) {
            float s[M][J];
            Core::load_scores(p, src, c0, s);
            Core::softmax_dropout(p, rng, row, c0, s, w, wd, keep);
        } else {
            Core::attention_weights(
                p, rng, row, c0, qs,
                [&](int m, int j) { return valid(j) ? ldg_cached(kv_row + Core::kv_rel(p, c0, m, 0, j)) : make_uint4(0, 0, 0, 0); },
                w, wd, keep);
        }

        // ---- value pass: d wd = dctx . v ; dV = wd * dctx ; d_bias_v += (sum_m wd) * dctx --------
        float dwd[M][J];
#pragma unroll
        for (int j = 0; j < J; ++j) {
            float dc[V];
            Vec<T>::unpack(dcraw[j], dc);
            uint4 raw[M];
#pragma unroll
            for (int m = 0; m < M; ++m) {
                if (PRELOAD_V) raw[m] = vraw[PRELOAD_V ? m : 0][PRELOAD_V ? j : 0];
                else raw[m] = valid(j) ? ldg_stream(kv_row + Core::kv_rel(p, c0, m, VHALF, j)) : make_uint4(0, 0, 0, 0);
            }
            float sum_wd = 0.f;
#pragma unroll
            for (int m = 0; m < M; ++m) {
                float f[V], dv[V];
                Vec<T>::unpack(raw[m], f);
                float a = 0.f;
#pragma unroll
                for (int v = 0; v < V; ++v) { a = fmaf(dc[v], f[v], a); dv[v] = wd[m][j] * dc[v]; }
                dwd[m][j] = a;
                sum_wd += wd[m][j];
                if (row_ok && valid(j)) stg_vec(dkv_row + Core::dkv_rel(p, c0, m, VHALF, j), Vec<T>::pack(dv));
            }
            if (row_ok && sums) strip_fma(acc_bv, j, lane, sum_wd, dc);
        }
        Core::head_reduce(p, dwd);

        // gradient arriving through the head-averaged weights (info['attention_weights'], and in
        // eval mode info['entropy'], reference aecf/AECFLayer.py:151-156, 538)
        if (p.d_pooled != nullptr || p.d_entropy != nullptr) {
            float dpw[M];
#pragma unroll
            for (int m = 0; m < M; ++m)
                dpw[m] = p.d_pooled ? __ldg(p.d_pooled + static_cast<size_t>(row) * M + m) : 0.f;
            if (p.d_entropy != nullptr) {
                float pw[M];
                Core::head_sum(p, c0, warp, lane, wd, xchg, pw);
                const float denom = static_cast<float>(p.H * p.R);
#pragma unroll
                for (int m = 0; m < M; ++m) pw[m] = pw[m] / denom;
                float raw;
                clamped_entropy<M>(pw, p.log_m, &raw);
                const bool inside = (raw >= 0.f) && (raw <= p.log_m);
                const float de = __ldg(p.d_entropy + row);
#pragma unroll
                for (int m = 0; m < M; ++m) dpw[m] += inside ? -(logf(pw[m]) + 1.0f) * de : 0.f;
            }
            const float h = static_cast<float>(p.H);
#pragma unroll
            for (int m = 0; m < M; ++m)
#pragma unroll
                for (int j = 0; j < J; ++j) dwd[m][j] += dpw[m] / h;
        }

        // ---- dropout and softmax backward ------------------------------------------------
        float ds[M][J];
#pragma unroll
        for (int j = 0; j < J; ++j) {
            float dot = 0.f;
#pragma unroll
            for (int m = 0; m < M; ++m) {
                float dw = dwd[m][j];
                if (DROP) dw = ((keep >> (m * J + j)) & 1u) ? dw / p.one_minus_p : 0.f;
                ds[m][j] = dw;
                dot = fmaf(w[m][j], dw, dot);
            }
            float sum_ds = 0.f;
#pragma unroll
            for (int m = 0; m < M; ++m) {
                ds[m][j] = w[m][j] * (ds[m][j] - dot);
                sum_ds += ds[m][j];
            }
            if (row_ok && valid(j) && sums) acc_sds[j * 32 + lane] += sum_ds;
            if (FOLD && p.rowsum != nullptr && row_ok) {     // the first lane of each head: [s | sum_m ds] of this sample
                const int c = c0 + 32 * j;
                if (valid(j) && (c & (p.G - 1)) == 0) {
                    float s_wd = 0.f;
#pragma unroll
                    for (int m = 0; m < M; ++m) s_wd += wd[m][j];
                    float* rs = p.rowsum + static_cast<size_t>(src) * (2 * p.HSP) + (c >> p.logG);
                    rs[0] = s_wd;
                    rs[p.HSP] = sum_ds;
                }
            }
        }

        if constexpr (FOLD) {
            // ---- score gradients next to dV: column D + head of the (row, m) line of d_kv; the first lane of
            // each head writes it, lanes 0 .. HSP-H-1 of the sample's first warp zero the padding columns
            if (row_ok) {
                T* line = reinterpret_cast<T*>(static_cast<char*>(p.d_kv) + static_cast<size_t>(src) * p.dkv_sb * sizeof(T)) + p.D;
#pragma unroll
                for (int j = 0; j < J; ++j) {
                    const int c = c0 + 32 * j;
                    if (valid(j) && (c & (p.G - 1)) == 0) {
                        const int head = c >> p.logG;
#pragma unroll
                        for (int m = 0; m < M; ++m) line[m * p.dkv_sm + head] = from_float<T>(ds[m][j]);
                    }
                }
                if (slice == 0 && lane < p.HSP - p.H) {
#pragma unroll
                    for (int m = 0; m < M; ++m) line[m * p.dkv_sm + p.H + lane] = from_float<T>(0.f);
                }
            }
        } else {
        // ---- key pass: dK = ds * (scale * q) ; dq += ds * k (K re-read: L1 hit) ------------------
#pragma unroll
        for (int j = 0; j < J; ++j) {
            uint4 raw[M];
#pragma unroll
            for (int m = 0; m < M; ++m)
                raw[m] = valid(j) ? ldg_cached(kv_row + Core::kv_rel(p, c0, m, 0, j)) : make_uint4(0, 0, 0, 0);
            float dq[V];
#pragma unroll
            for (int v = 0; v < V; ++v) dq[v] = 0.f;
            float sum_ds = 0.f;
#pragma unroll
            for (int m = 0; m < M; ++m) {
                float f[V], dk[V];
                Vec<T>::unpack(raw[m], f);
#pragma unroll
                for (int v = 0; v < V; ++v) {
                    dk[v] = ds[m][j] * qs[j][v];
                    dq[v] = fmaf(ds[m][j], f[v], dq[v]);
                }
                sum_ds += ds[m][j];
                if (row_ok && valid(j)) stg_vec(dkv_row + Core::dkv_rel(p, c0, m, 0, j), Vec<T>::pack(dk));
            }
            if (row_ok) {
                if (p.q_shared) {
#pragma unroll
                    for (int q4 = 0; q4 < Q4; ++q4) {
                        float4 a = acc_q[(j * Q4 + q4) * 32 + lane];
                        a.x += dq[4 * q4]; a.y += dq[4 * q4 + 1]; a.z += dq[4 * q4 + 2]; a.w += dq[4 * q4 + 3];
                        acc_q[(j * Q4 + q4) * 32 + lane] = a;
                    }
                } else {
                    // per-row query: d_q[row] = scale * dq; the strip accumulates d_bias_k = sum dK instead
                    float o[V];
#pragma unroll
                    for (int v = 0; v < V; ++v) o[v] = dq[v] * p.scale;
                    if (valid(j))
                        stg_vec(static_cast<char*>(p.d_q) + static_cast<size_t>(row) * p.D * sizeof(T)
                                    + Core::lane_bytes(p, c0) + Core::col_bytes(p, c0, j), Vec<T>::pack(o));
                    strip_fma(acc_q, j, lane, sum_ds, qs[j]);
                }
            }
        }
        }   // !FOLD
    }

    // ---- fold the warps' strips in a fixed order into this CTA's partial [3][D] -----------------
    // partial[0] = d_q (shared query, unscaled)   partial[1] = d_bias_v   partial[2] = d_bias_k
    if (!sums) return;
    __syncthreads();
    const int D = p.D;
    float* out = p.partials + static_cast<size_t>(blockIdx.x) * 3 * D;
    const float* strips = smem + POOL_WARPS * M;
    for (int i = threadIdx.x + (FOLD ? D : 0); i < 3 * D; i += blockDim.x) {     // folded: there is no d_q third
        const int which = i / D, d = i - which * D;
        const int rc = d / V, v = d - rc * V;
        const int c = Core::virtual_chunk(p, rc);                 // the strips are laid out by lane, i.e. by virtual chunk
        const int sl = c / Core::CPW, cl = c - sl * Core::CPW;
        const int j = cl >> 5, ln = cl & 31;
        const int idx = ((j * Q4 + (v >> 2)) * 32 + ln) * 4 + (v & 3);
        float s = 0.f;
        for (int smp = 0; smp < p.SPC; ++smp) {
            const float* st = strips + (smp * p.WPS + sl) * Smem::PER_WARP;
            if (which == 1) s += st[Smem::ACC + idx];
            else if (which == 0) s += p.q_shared ? st[idx] : 0.f;
            else s += p.q_shared ? st[2 * Smem::ACC + j * 32 + ln] : st[idx];
        }
        if (which == 2 && p.q_shared) s *= __ldg(static_cast<const float*>(p.q) + d) * p.scale;
        out[i] = s;
    }
}

}  // namespace aecf
