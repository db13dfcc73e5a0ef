// Fused pool kernels for several fusion queries per sample (target length S > 1).
//
// The reference accepts any [B, S, D] query (aecf/AECFLayer.py:415, torch/nn/functional.py:6632-6659): every
// (b, s) pair is a row of its own for the scores, softmax, dropout, head mean and the CurriculumMasking stage,
// and the S rows of a sample share its M projected keys and values.  The fusion hot path has S == 1 (one fusion
// token, pool_fwd.cuh / pool_bwd.cuh); these kernels cover the rest of the reference's surface with the same
// building blocks (pool_core.cuh, masking_stage) and the same arithmetic, not the same tuning:
//   forward   one warp slice per (b, s) row; the S rows of a sample re-read its kv through L1/L2
//   backward  persistent over SAMPLES; a warp slice walks the S queries of its sample and sums dK / dV over them
//             in fp32 registers, so d_kv is written once and the GEMMs that follow are those of S == 1
// Row conventions: info outputs, d_pooled, d_entropy and the Philox row use the index b*S + s (the host passes
// rng.row0 = row0 * S); q, ctx, d_ctx and d_q rows sit at b*q_rb + s*q_rs (batch-first (S, 1), sequence-first
// (1, B)).  The additive score bias comes in MultiQuery (PoolParams::bias is null in this mode).
#pragma once

#include "pool_bwd.cuh"
#include "pool_fwd.cuh"

namespace aecf {

// + additive mask of row (b, s), torch/nn/functional.py:6638 baddbmm(attn_mask, q, k^T)
template <typename Core, int M, int J>
__device__ __forceinline__ void add_score_bias(const PoolParams& p, const MultiQuery& mq, long long b, int s, int c0,
                                               float (&sc)[M][J]) {
    if (mq.bias == nullptr) return;
    int head[J];
    Core::heads_of(p, c0, head);
#pragma unroll
    for (int j = 0; j < J; ++j) {
        const float* base = mq.bias + static_cast<size_t>(b) * mq.bias_sb + static_cast<size_t>(s) * mq.bias_ss
                            + static_cast<size_t>(head[j]) * mq.bias_sh;
#pragma unroll
        for (int m = 0; m < M; ++m) sc[m][j] += __ldg(base + m);
    }
}

// PAD: the padded lane map (pool_core.cuh).
template <typename T, int M, int J, bool DROP, bool PAD>
__global__ void __launch_bounds__(POOL_WARPS * 32)
pool_fwd_multi_kernel(const PoolParams p, const MultiQuery mq) {
    using Core = PoolCore<T, M, J, DROP, PAD>;
    constexpr int V = Core::V;
    __shared__ float xchg[POOL_WARPS * M];
    __shared__ float head_sums[POOL_WARPS * M];       // [row slot][m], written by the slice-0 warps
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int slice = warp % p.WPS;
    const int slot = warp / p.WPS;
    const long long n = p.B * mq.S;                   // rows (b, s), b-major
    const long long first = static_cast<long long>(blockIdx.x) * p.SPC;
    const bool row_ok = first + slot < n;
    const long long row = row_ok ? first + slot : n - 1;      // tail warps recompute the last row, store nothing
    const long long b = row / mq.S;
    const int s = static_cast<int>(row - b * mq.S);
    const long long qrow = b * mq.q_rb + s * mq.q_rs;
    const int c0 = slice * Core::CPW + lane;
    pdl_wait();
    const RngKey rng = effective_rng(p.rng, p.rng_state);

    const char* kv_row = static_cast<const char*>(p.kv) + Core::row_offset(p, b, c0);
    auto load_kv = [&](int m, int half, int j) -> uint4 {
        return Core::valid(p, c0, j) ? ldg_cached(kv_row + Core::kv_rel(p, c0, m, half, j)) : make_uint4(0, 0, 0, 0);
    };

    float qs[J][V];
    Core::load_query(p, qrow, c0, qs);
    float sc[M][J], w[M][J], wd[M][J];
    unsigned keep;
    Core::key_scores(p, qs, [&](int m, int j) { return load_kv(m, 0, j); }, sc);
    add_score_bias<Core, M, J>(p, mq, b, s, c0, sc);
    Core::softmax_dropout(p, rng, row, c0, sc, w, wd, keep);

    // ---- weighted value sum (torch/nn/functional.py:6647) ---------------------------------
    float acc[J][V];
#pragma unroll
    for (int j = 0; j < J; ++j)
#pragma unroll
        for (int v = 0; v < V; ++v) acc[j][v] = 0.f;
#pragma unroll
    for (int m = 0; m < M; ++m)
#pragma unroll
        for (int j = 0; j < J; ++j) {
            float f[V];
            Vec<T>::unpack(load_kv(m, 1, j), f);
#pragma unroll
            for (int v = 0; v < V; ++v) acc[j][v] = fmaf(wd[m][j], f[v], acc[j][v]);
        }
    if (row_ok) {
        char* ctx = static_cast<char*>(p.ctx) + static_cast<size_t>(qrow) * p.D * sizeof(T) + Core::lane_bytes(p, c0);
        if constexpr (PAD) {
#pragma unroll
            for (int j = 0; j < J; ++j)
                if (Core::valid(p, c0, j)) stg_vec(ctx + Core::col_bytes(p, c0, j), Vec<T>::pack(acc[j]));
        } else {    // the original spelling (see PoolCore::load_row)
#pragma unroll
            for (int j = 0; j < J; ++j)
                if (c0 + 32 * j < p.NC) stg_vec(ctx + j * 512, Vec<T>::pack(acc[j]));
        }
    }

    // ---- head sums of the post-dropout weights -> shared memory; warp 0 finishes the CTA's rows -----
    float total[M];
    Core::head_sum(p, c0, warp, lane, wd, xchg, total);
    if (slice == 0 && lane == 0) {
#pragma unroll
        for (int m = 0; m < M; ++m) head_sums[slot * M + m] = total[m];
    }
    __syncthreads();
    if (warp != 0) return;

    // ---- head mean (torch/nn/functional.py:6657-6659) and CurriculumMasking, one row per lane -------
    const long long my_row = first + lane;
    if (lane >= p.SPC || my_row >= n) return;
    const float denom = static_cast<float>(p.H * p.R);
    float pw[M], mw[M];
#pragma unroll
    for (int m = 0; m < M; ++m) pw[m] = head_sums[lane * M + m] / denom;
    float entropy, mask_rate;
    unsigned bits;
    masking_stage<M>(p, rng, my_row, pw, mw, entropy, mask_rate, bits);
    store_info<M>(p, my_row, pw, mw, entropy, mask_rate, bits);
}

// Backward.  Same closed form as pool_bwd_kernel (SURVEY.md Appendix B) per (b, s) row; dK and dV of a sample are
// the sums over its S rows, d_q is per row.  The strips accumulate d_bias_v and d_bias_k (= sum dK) as in the
// per-row-query mode of pool_bwd_kernel, and are folded into partials in the same layout, so the same finalize
// kernel applies.  One CTA per SM: the fp32 dK / dV accumulators take 2*M*J*V registers per lane.
template <typename T, int M, int J, bool DROP, bool PAD>
__global__ void __launch_bounds__(POOL_WARPS * 32, 1)
pool_bwd_multi_kernel(const PoolParams p, const MultiQuery mq) {
    using Core = PoolCore<T, M, J, DROP, PAD>;
    using Smem = BwdSmem<J, Core::V>;
    constexpr int V = Core::V;
    constexpr int Q4 = V / 4;

    AECF_DYNAMIC_SMEM_ALIGNED16(float, smem);
    float* xchg = smem;                                               // [POOL_WARPS][M]
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    float* strip = smem + POOL_WARPS * M + warp * Smem::PER_WARP;     // this warp's accumulators
    float4* acc_bk = reinterpret_cast<float4*>(strip);                // [J][Q4][32]  sum dK
    float4* acc_bv = reinterpret_cast<float4*>(strip + Smem::ACC);    // [J][Q4][32]  sum dV
    for (int i = lane; i < Smem::PER_WARP; i += 32) strip[i] = 0.f;
    __syncwarp();
    pdl_wait();
    const RngKey rng = effective_rng(p.rng, p.rng_state);

    const int slice = warp % p.WPS;
    const int c0 = slice * Core::CPW + lane;
    auto valid = [&](int j) { return Core::valid(p, c0, j); };

    const long long stride = static_cast<long long>(gridDim.x) * p.SPC;
    for (long long base = static_cast<long long>(blockIdx.x) * p.SPC; base < p.B; base += stride) {
        const long long b_raw = base + warp / p.WPS;
        const bool row_ok = b_raw < p.B;
        const long long b = row_ok ? b_raw : p.B - 1;
        const char* kv_row = static_cast<const char*>(p.kv) + Core::row_offset(p, b, c0);
        char* dkv_row = static_cast<char*>(p.d_kv) + Core::drow_offset(p, b, c0);
        auto load_kv = [&](int m, int half, int j) -> uint4 {
            return valid(j) ? ldg_cached(kv_row + Core::kv_rel(p, c0, m, half, j)) : make_uint4(0, 0, 0, 0);
        };

        float dk_acc[M][J][V], dv_acc[M][J][V];
#pragma unroll
        for (int m = 0; m < M; ++m)
#pragma unroll
            for (int j = 0; j < J; ++j)
#pragma unroll
                for (int v = 0; v < V; ++v) { dk_acc[m][j][v] = 0.f; dv_acc[m][j][v] = 0.f; }

        for (int s = 0; s < mq.S; ++s) {
            const long long row = b * mq.S + s;
            const long long qrow = b * mq.q_rb + s * mq.q_rs;
            float qs[J][V];
            Core::load_query(p, qrow, c0, qs);
            uint4 dcraw[J];
            Core::load_row(p, p.d_ctx, qrow, c0, dcraw);

            float sc[M][J], w[M][J], wd[M][J];
            unsigned keep;
            Core::key_scores(p, qs, [&](int m, int j) { return load_kv(m, 0, j); }, sc);
            add_score_bias<Core, M, J>(p, mq, b, s, c0, sc);
            Core::softmax_dropout(p, rng, row, c0, sc, w, wd, keep);

            // ---- value pass: d wd = dctx . v ; dV += wd * dctx ; d_bias_v += (sum_m wd) * dctx --------
            float dwd[M][J];
#pragma unroll
            for (int j = 0; j < J; ++j) {
                float dc[V];
                Vec<T>::unpack(dcraw[j], dc);
                float sum_wd = 0.f;
#pragma unroll
                for (int m = 0; m < M; ++m) {
                    float f[V];
                    Vec<T>::unpack(load_kv(m, 1, j), f);
                    float a = 0.f;
#pragma unroll
                    for (int v = 0; v < V; ++v) {
                        a = fmaf(dc[v], f[v], a);
                        dv_acc[m][j][v] = fmaf(wd[m][j], dc[v], dv_acc[m][j][v]);
                    }
                    dwd[m][j] = a;
                    sum_wd += wd[m][j];
                }
                if (row_ok) strip_fma(acc_bv, j, lane, sum_wd, dc);
            }
            Core::head_reduce(p, dwd);

            // gradient arriving through the head-averaged weights (info['attention_weights'], and in eval mode
            // info['entropy'], reference aecf/AECFLayer.py:151-156, 538)
            if (p.d_pooled != nullptr || p.d_entropy != nullptr) {
                float dpw[M];
#pragma unroll
                for (int m = 0; m < M; ++m)
                    dpw[m] = p.d_pooled ? __ldg(p.d_pooled + static_cast<size_t>(row) * M + m) : 0.f;
                if (p.d_entropy != nullptr) {
                    float pw[M];
                    Core::head_sum(p, c0, warp, lane, wd, xchg, pw);      // CTA-uniform: every warp walks all S rows
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
#pragma unroll
                for (int m = 0; m < M; ++m) ds[m][j] = w[m][j] * (ds[m][j] - dot);
            }

            // ---- key pass: dK += ds * (scale * q) ; d_q[row] = scale * sum_m ds * k (K re-read: L1 hit) ------
#pragma unroll
            for (int j = 0; j < J; ++j) {
                float dq[V];
#pragma unroll
                for (int v = 0; v < V; ++v) dq[v] = 0.f;
                float sum_ds = 0.f;
#pragma unroll
                for (int m = 0; m < M; ++m) {
                    float f[V];
                    Vec<T>::unpack(load_kv(m, 0, j), f);
#pragma unroll
                    for (int v = 0; v < V; ++v) {
                        dk_acc[m][j][v] = fmaf(ds[m][j], qs[j][v], dk_acc[m][j][v]);
                        dq[v] = fmaf(ds[m][j], f[v], dq[v]);
                    }
                    sum_ds += ds[m][j];
                }
                if (row_ok) {
                    float o[V];
#pragma unroll
                    for (int v = 0; v < V; ++v) o[v] = dq[v] * p.scale;
                    if (valid(j))
                        stg_vec(static_cast<char*>(p.d_q) + static_cast<size_t>(qrow) * p.D * sizeof(T)
                                    + Core::lane_bytes(p, c0) + Core::col_bytes(p, c0, j), Vec<T>::pack(o));
                    strip_fma(acc_bk, j, lane, sum_ds, qs[j]);          // d_bias_k = sum dK
                }
            }
        }

        if (row_ok) {
#pragma unroll
            for (int m = 0; m < M; ++m)
#pragma unroll
                for (int j = 0; j < J; ++j)
                    if (valid(j)) {
                        stg_vec(dkv_row + Core::dkv_rel(p, c0, m, 0, j), Vec<T>::pack(dk_acc[m][j]));
                        stg_vec(dkv_row + Core::dkv_rel(p, c0, m, 1, j), Vec<T>::pack(dv_acc[m][j]));
                    }
        }
    }

    // ---- fold the warps' strips in a fixed order into this CTA's partial [3][D] (layout of pool_bwd_kernel:
    // partial[0] unused with per-row queries, partial[1] = d_bias_v, partial[2] = d_bias_k) -----------------
    __syncthreads();
    const int D = p.D;
    float* out = p.partials + static_cast<size_t>(blockIdx.x) * 3 * D;
    const float* strips = smem + POOL_WARPS * M;
    for (int i = threadIdx.x; i < 3 * D; i += blockDim.x) {
        const int which = i / D, d = i - which * D;
        const int rc = d / V, v = d - rc * V;
        const int c = Core::virtual_chunk(p, rc);
        const int sl = c / Core::CPW, cl = c - sl * Core::CPW;
        const int j = cl >> 5, ln = cl & 31;
        const int idx = ((j * Q4 + (v >> 2)) * 32 + ln) * 4 + (v & 3);
        float t = 0.f;
        if (which != 0) {
            for (int smp = 0; smp < p.SPC; ++smp)
                t += strips[(smp * p.WPS + sl) * Smem::PER_WARP + (which == 1 ? Smem::ACC : 0) + idx];
        }
        out[i] = t;
    }
}

}  // namespace aecf
