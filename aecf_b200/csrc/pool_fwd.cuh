// Fused pool forward: one launch for
//   scale -> per-head scores -> softmax -> dropout -> weighted value sum -> head mean
//   -> CurriculumMasking (renormalise, entropy, keep-prob, Philox mask, min_active repair,
//      renormalise, mask_rate).
// Replaces torch/nn/functional.py:6632-6647, 6657-6659 and reference aecf/AECFLayer.py:130-283.
// HBM-bound: algorithmic bytes per sample = s*(2*M*D + D) + 4*(2*M + 2)  (SURVEY.md section 8d).
//
// Structure.  The data phase is warp-per-sample-slice (pool_core.cuh) and issues every load of
// the slice before any arithmetic.  The masking stage is a few dozen scalar operations per SAMPLE:
// run by the warp that owns the sample it would cost a full warp instruction per scalar op, so the
// warps hand their head sums to shared memory and warp 0 finishes all of the CTA's samples at once,
// one sample per lane (r1 profile: 1 160 -> ~400 warp instructions per sample).
#pragma once

#include "pool_core.cuh"

namespace aecf {

// CurriculumMasking.forward for one sample, exact IEEE arithmetic (reference aecf/AECFLayer.py:130-283).
template <int M>
__device__ __forceinline__ void masking_stage(const PoolParams& p, const RngKey& rng, long long row, const float (&pw)[M],
                                              float (&mw)[M], float& entropy, float& mask_rate, unsigned& bits) {
    entropy = 0.f;
    mask_rate = 0.f;
    bits = (1u << M) - 1u;
#pragma unroll
    for (int m = 0; m < M; ++m) mw[m] = pw[m];
    if (!p.masking) return;
    if (p.masking == 2) {                                             // eval mode, :150-156
        entropy = clamped_entropy<M>(pw, p.log_m);
        return;
    }
    if (M <= 1) return;                                               // :159-167: zeros, weights unchanged
    float wn[M];
    float total = 0.f;
#pragma unroll
    for (int m = 0; m < M; ++m) {                                     // :170-176 NaN/Inf scrub
        wn[m] = (fabsf(pw[m]) <= 3.402823466e38f) ? pw[m] : 0.f;
        total = __fadd_rn(total, wn[m]);
    }
    const bool degenerate = total < 1e-8f;                            // :178 (the _eps buffer)
#pragma unroll
    for (int m = 0; m < M; ++m) wn[m] = degenerate ? (1.0f / M) : wn[m] / total;   // :181-184
    entropy = clamped_entropy<M>(wn, p.log_m);                        // :190
    const float norm_entropy = fminf(fmaxf(entropy / p.log_m, 0.f), 1.f);          // :192
    // mul then sub, each rounded (no FMA contraction): the mask threshold must match bit for bit
    const float keep_prob =
        fminf(fmaxf(__fsub_rn(1.0f, __fmul_rn(p.base_mask_prob, norm_entropy)), 0.f), 1.f);   // :197-201

    float u[(M + 3) / 4 * 4];
#pragma unroll
    for (int blk = 0; blk < (M + 3) / 4; ++blk) {
        float u4[4];
        draw4(rng, static_cast<unsigned long long>(row), STREAM_MASK, 0u, blk, u4);
#pragma unroll
        for (int i = 0; i < 4; ++i) u[4 * blk + i] = u4[i];
    }
    bits = 0u;
    int active = 0;
#pragma unroll
    for (int m = 0; m < M; ++m) {                                     // :204 bernoulli(keep_prob)
        const bool k = u[m] <= keep_prob;
        bits |= k ? (1u << m) : 0u;
        active += k ? 1 : 0;
    }
    const int need = min(p.min_active, M);                            // :207
    if (active < need) {                                              // :209-260: REPLACE by the top-`need` set
        bits = 0u;
#pragma unroll
        for (int i = 0; i < M; ++i) {
            int rank = 0;                                             // entries that beat i (ties: lower index wins)
#pragma unroll
            for (int j = 0; j < M; ++j) rank += (wn[j] > wn[i] || (wn[j] == wn[i] && j < i)) ? 1 : 0;
            bits |= (rank < need) ? (1u << i) : 0u;
        }
        active = need;
    }
    float kept_sum = 0.f;
#pragma unroll
    for (int m = 0; m < M; ++m) {                                     // :263-264
        mw[m] = ((bits >> m) & 1u) ? wn[m] : 0.f;
        kept_sum = __fadd_rn(kept_sum, mw[m]);
    }
    const bool valid = kept_sum > 1e-8f;                              // :267
#pragma unroll
    for (int m = 0; m < M; ++m) mw[m] = valid ? mw[m] / kept_sum : wn[m];          // :268-272
    mask_rate = __fsub_rn(1.0f, static_cast<float>(active) / static_cast<float>(M));   // :275
}

// The info outputs of one row, as masking_stage left them.
template <int M>
__device__ __forceinline__ void store_info(const PoolParams& p, long long row, const float (&pw)[M], const float (&mw)[M],
                                           float entropy, float mask_rate, unsigned bits) {
#pragma unroll
    for (int m = 0; m < M; ++m) {
        p.pooled[static_cast<size_t>(row) * M + m] = pw[m];
        if (p.masked) p.masked[static_cast<size_t>(row) * M + m] = mw[m];
    }
    if (p.entropy) p.entropy[row] = entropy;
    if (p.mask_rate) p.mask_rate[row] = mask_rate;
    if (p.mask_bits) p.mask_bits[row] = static_cast<uint8_t>(bits);
}

// FOLD: folded key projection -- kv holds the values only and the scores come precomputed (pool_core.cuh).
// PAD: the padded lane map (pool_core.cuh).
template <typename T, int M, int J, bool DROP, bool FOLD, bool PAD>
__global__ void __launch_bounds__(POOL_WARPS * 32)
pool_fwd_kernel(const PoolParams p) {
    using Core = PoolCore<T, M, J, DROP, PAD>;
    constexpr int V = Core::V;
    constexpr int VHALF = FOLD ? 0 : 1;                 // which D-wide half of a kv row holds the values
    __shared__ float xchg[POOL_WARPS * M];
    __shared__ float head_sums[POOL_WARPS * M];       // [sample slot][m], written by the slice-0 warps
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int slice = warp % p.WPS;
    const int slot = warp / p.WPS;
    const long long row0 = static_cast<long long>(blockIdx.x) * p.SPC;
    const bool row_ok = row0 + slot < p.B;
    const long long row = row_ok ? row0 + slot : p.B - 1;   // tail warps recompute the last row, store nothing
    const int c0 = slice * Core::CPW + lane;
    pdl_wait();
    const RngKey rng = effective_rng(p.rng, p.rng_state);
    const long long src = source_row(p, row);              // where the row's sample lives in kv / scores / ctx

    const char* kv_row = static_cast<const char*>(p.kv) + Core::row_offset(p, src, c0);
    auto load_kv = [&](int m, int half, int j) -> uint4 {
        return Core::valid(p, c0, j) ? ldg_stream(kv_row + Core::kv_rel(p, c0, m, half, j)) : make_uint4(0, 0, 0, 0);
    };

    // Issue the value loads first when they fit in registers: the whole slice is then in flight
    // before any arithmetic starts (12 x 16 B per lane at M=3, D=512 bf16).
    constexpr bool PRELOAD_V = (M * J <= 8);
    uint4 vraw[PRELOAD_V ? M : 1][PRELOAD_V ? J : 1];
    if (PRELOAD_V) {
#pragma unroll
        for (int m = 0; m < M; ++m)
#pragma unroll
            for (int j = 0; j < J; ++j) vraw[PRELOAD_V ? m : 0][PRELOAD_V ? j : 0] = load_kv(m, VHALF, j);
    }

    float w[M][J], wd[M][J];
    unsigned keep;
    if constexpr (FOLD) {
        float s[M][J];
        Core::load_scores(p, src, c0, s);
        Core::softmax_dropout(p, rng, row, c0, s, w, wd, keep);
    } else {
        float qs[J][V];
        Core::load_query(p, row, c0, qs);
        Core::attention_weights(p, rng, row, c0, qs, [&](int m, int j) { return load_kv(m, 0, j); }, w, wd, keep);
    }

    // ---- weighted value sum (torch/nn/functional.py:6647) ---------------------------------
    float acc[J][V];
#pragma unroll
    for (int j = 0; j < J; ++j)
#pragma unroll
        for (int v = 0; v < V; ++v) acc[j][v] = 0.f;
#pragma unroll
    for (int m = 0; m < M; ++m) {
        uint4 raw[J];
#pragma unroll
        for (int j = 0; j < J; ++j)
            raw[j] = PRELOAD_V ? vraw[PRELOAD_V ? m : 0][PRELOAD_V ? j : 0] : load_kv(m, VHALF, j);
#pragma unroll
        for (int j = 0; j < J; ++j) {
            float f[V];
            Vec<T>::unpack(raw[j], f);
#pragma unroll
            for (int v = 0; v < V; ++v) acc[j][v] = fmaf(wd[m][j], f[v], acc[j][v]);
        }
    }
    if (row_ok) {
        char* ctx = static_cast<char*>(p.ctx) + static_cast<size_t>(src) * p.D * sizeof(T) + Core::lane_bytes(p, c0);
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

    // ---- head sums of the post-dropout weights -> shared memory ----------------------------------
    float total[M];
    Core::head_sum(p, c0, warp, lane, wd, xchg, total);
    if (slice == 0 && lane == 0) {
#pragma unroll
        for (int m = 0; m < M; ++m) head_sums[slot * M + m] = total[m];
    }
#ifdef AECF_CUDA_EMU
    if (warp != 0) { cuda_emu::named_barrier(1, POOL_WARPS * 32, false); return; }
    cuda_emu::named_barrier(1, POOL_WARPS * 32, true);
#else
    if (warp != 0) {                                   // hand over and retire; warp 0 finishes the CTA's samples
        asm volatile("bar.arrive 1, %0;" :: "n"(POOL_WARPS * 32) : "memory");
        return;
    }
    asm volatile("bar.sync 1, %0;" :: "n"(POOL_WARPS * 32) : "memory");
#endif

    // ---- head mean (torch/nn/functional.py:6657-6659) and CurriculumMasking, one sample per lane -------
    const long long my_row = row0 + lane;
    if (lane >= p.SPC || my_row >= p.B) return;
    const float denom = static_cast<float>(p.H * p.R);     // R copies of each head when G > 32 (R = 2^k: exact)
    float pw[M], mw[M];
#pragma unroll
    for (int m = 0; m < M; ++m) pw[m] = head_sums[lane * M + m] / denom;
    float entropy, mask_rate;
    unsigned bits;
    masking_stage<M>(p, rng, my_row, pw, mw, entropy, mask_rate, bits);
    store_info<M>(p, my_row, pw, mw, entropy, mask_rate, bits);
}

// ---- streaming variant (one warp owns a whole sample, WPS == 1): the headline path ----------------------
// Persistent warps, each on a contiguous block of rows.  The next row's K/V chunks are copied
// global -> shared with cp.async (16 B per lane, no register staging) while the current row is being
// reduced, so every warp keeps one full sample (6 KB at M=3, D=512 bf16) in flight at all times and the
// arithmetic never waits on HBM.  Head sums of up to 32 consecutive rows stay in lane registers (lane i
// keeps row i); the masking stage then runs once per 32 rows with one row per lane.
// DENSE (folded only): every lane owns J valid chunks (D = 32 J chunks exactly) and a sample's M value rows are contiguous,
// so chunk (m, j) sits at the compile-time offset (m J + j) * 512 and no access needs a validity test -- 50 of the generic
// kernel's 493 instructions per sample were address arithmetic and tests of exactly that (ncu source page, r2 run 26).
// PAD (padded lane map) is never DENSE: each lane copies exactly its own valid chunks, at their real addresses, into its own
// ring slots and reads back only those, so the ring keeps its own-copies-only wait.
template <typename T, int M, int J, bool DROP, bool FOLD, bool DENSE, bool PAD>
__global__ void __launch_bounds__((FOLD && J <= 2) ? 768 : 512, 1)
pool_fwd_stream_kernel(const PoolParams p, const long long rows_per_warp) {
    static_assert(!(DENSE && PAD), "the dense specialisation assumes the power-of-two lane map");
    using Core = PoolCore<T, M, J, DROP, PAD>;
    constexpr int V = Core::V;
    constexpr int HALVES = FOLD ? 1 : 2;                // folded: only the values are staged
    constexpr int VHALF = FOLD ? 0 : 1;
    constexpr int CH = M * HALVES * J;                  // 16-byte chunks per lane per sample
    AECF_DYNAMIC_SMEM(uint4, ring);                     // [warps][2 stages][CH][32 lanes]
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const long long gw = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + warp;
    const long long row_begin = min(p.B, gw * rows_per_warp);
    const long long row_end = min(p.B, row_begin + rows_per_warp);
    // fused entropy_loss: every warp, with or without rows, hands in a partial sum at the end (no block-level barrier:
    // a shared-memory counter elects the CTA's last warp)
    // (the two variables live BEHIND the ring in dynamic shared memory: a static __shared__ array would push the ring off
    // its 128-byte alignment and every 512-byte warp access of the ring would touch five lines instead of four -- r2 run 4
    // measured 50 -> 58 us for exactly that)
    float* cta_loss = reinterpret_cast<float*>(ring + static_cast<size_t>(blockDim.x >> 5) * 2 * CH * 32);   // [32]
    unsigned& cta_done = *reinterpret_cast<unsigned*>(cta_loss + 32);
    if (p.loss_out != nullptr && threadIdx.x == 0) cta_done = 0u;
    if (p.loss_out != nullptr) __syncthreads();         // the only block-level barrier, before any warp can finish
    float loss_acc = 0.f;                               // this lane's rows: sum of (scrubbed entropy - target)^2
    uint4* my = ring + static_cast<size_t>(warp) * 2 * CH * 32;
    const int c0 = lane;
    const char* kv = static_cast<const char*>(p.kv);
    pdl_wait();
    const RngKey rng = effective_rng(p.rng, p.rng_state);

    auto prefetch = [&](long long row, int stage) {
        const char* src = kv + Core::row_offset(p, row, c0);
#pragma unroll
        for (int m = 0; m < M; ++m)
#pragma unroll
            for (int half = 0; half < HALVES; ++half)
#pragma unroll
                for (int j = 0; j < J; ++j)
                    if (DENSE || Core::valid(p, c0, j))
                        cp_async16(&my[(stage * CH + (m * HALVES + half) * J + j) * 32 + lane],
                                   src + (DENSE ? (m * J + j) * 512 : Core::kv_rel(p, c0, m, half, j)));
        cp_async_commit();
    };
    if (row_begin < row_end) prefetch(row_begin, 0);

    float qs[J][V];
    if (!FOLD && p.q_shared) Core::load_query(p, 0, c0, qs);
    float s_next[M][J];                                 // folded: the next row's scores, loaded one row ahead
    if constexpr (FOLD) {
        if (row_begin < row_end) Core::load_scores(p, row_begin, c0, s_next);
    }
    const float denom = static_cast<float>(p.H * p.R);
    float mine[M];                                      // head sums of the row this lane will finish
#pragma unroll
    for (int m = 0; m < M; ++m) mine[m] = 0.f;

    int it = 0;
    for (long long row = row_begin; row < row_end; ++row, ++it) {
        const int stage = it & 1;
        if (row + 1 < row_end) prefetch(row + 1, stage ^ 1);
        else cp_async_commit();                         // empty group keeps the wait count uniform
        if (!FOLD && !p.q_shared) Core::load_query(p, row, c0, qs);
        float s[M][J];
        if constexpr (FOLD) {
#pragma unroll
            for (int m = 0; m < M; ++m)
#pragma unroll
                for (int j = 0; j < J; ++j) s[m][j] = s_next[m][j];
            if (row + 1 < row_end) Core::load_scores(p, row + 1, c0, s_next);
        }
        cp_async_wait<1>();                             // this row's chunks have landed (own copies only)
        auto staged = [&](int m, int half, int j) -> uint4 {
            return (DENSE || Core::valid(p, c0, j)) ? my[(stage * CH + (m * HALVES + half) * J + j) * 32 + lane] : make_uint4(0, 0, 0, 0);
        };

        float w[M][J], wd[M][J];
        unsigned keep;
        if constexpr (FOLD) Core::softmax_dropout(p, rng, row, c0, s, w, wd, keep);
        else Core::attention_weights(p, rng, row, c0, qs, [&](int m, int j) { return staged(m, 0, j); }, w, wd, keep);

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
                Vec<T>::unpack(staged(m, VHALF, j), f);
#pragma unroll
                for (int v = 0; v < V; ++v) acc[j][v] = fmaf(wd[m][j], f[v], acc[j][v]);
            }
        char* ctx = static_cast<char*>(p.ctx) + static_cast<size_t>(row) * p.D * sizeof(T) + Core::lane_bytes(p, c0);
        if constexpr (PAD) {
#pragma unroll
            for (int j = 0; j < J; ++j)
                if (Core::valid(p, c0, j)) stg_vec(ctx + Core::col_bytes(p, c0, j), Vec<T>::pack(acc[j]));
        } else {    // the original spelling (see PoolCore::load_row)
#pragma unroll
            for (int j = 0; j < J; ++j)
                if (DENSE || c0 + 32 * j < p.NC) stg_vec(ctx + j * 512, Vec<T>::pack(acc[j]));
        }

        float total[M];
        Core::head_sum_partial(p, c0, wd, total);       // WPS == 1: the warp holds every head
#pragma unroll
        for (int m = 0; m < M; ++m) mine[m] = (lane == (it & 31)) ? total[m] : mine[m];

        if ((it & 31) == 31 || row + 1 == row_end) {    // finish up to 32 rows, one per lane
            const long long first = row - (it & 31);
            const long long my_row = first + lane;
            if (my_row <= row) {
                float pw[M], mw[M];
#pragma unroll
                for (int m = 0; m < M; ++m) pw[m] = mine[m] / denom;
                float entropy, mask_rate;
                unsigned bits;
                masking_stage<M>(p, rng, my_row, pw, mw, entropy, mask_rate, bits);
                store_info<M>(p, my_row, pw, mw, entropy, mask_rate, bits);
                if (p.loss_out != nullptr) {            // reference aecf/AECFLayer.py:299-311, the per-sample term
                    bool fin;
                    const float d = scrub_entropy(entropy, &fin) - p.loss_target;
                    loss_acc = fmaf(d, d, loss_acc);
                }
            }
            __syncwarp();
        }
    }
    if (p.loss_out == nullptr) return;
    // ---- entropy_loss = max(0, mean_b (.)^2): lanes -> warp (xor shuffles), warps -> CTA and CTAs -> result in INDEX
    // order by whoever finishes last: the value does not depend on the finishing order
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) loss_acc += __shfl_xor_sync(FULL_MASK, loss_acc, off);
    const int warps = blockDim.x >> 5;
    unsigned last_warp = 0u;
    if (lane == 0) {
        cta_loss[warp] = loss_acc;
        __threadfence_block();
        last_warp = (atomicAdd(&cta_done, 1u) == static_cast<unsigned>(warps - 1)) ? 1u : 0u;
    }
    last_warp = __shfl_sync(FULL_MASK, last_warp, 0);
    if (!last_warp) return;
    __threadfence_block();
    unsigned last_cta = 0u;
    if (lane == 0) {
        float s = 0.f;
        for (int w = 0; w < warps; ++w) s += cta_loss[w];
        p.loss_partials[blockIdx.x] = s;
        __threadfence();
        last_cta = (atomicAdd(p.loss_ticket, 1u) == gridDim.x - 1) ? 1u : 0u;
    }
    last_cta = __shfl_sync(FULL_MASK, last_cta, 0);
    if (!last_cta) return;
    __threadfence();
    float s = 0.f;
    for (unsigned b = lane; b < gridDim.x; b += 32) s += p.loss_partials[b];     // lane l: CTAs l, l + 32, ... in order
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(FULL_MASK, s, off);
    if (lane == 0) {
        p.loss_out[0] = fmaxf(s / static_cast<float>(p.B), 0.f);                 // .mean().clamp_(min=0)
        *p.loss_ticket = 0u;                                                     // re-armed for the next launch
    }
}

}  // namespace aecf
