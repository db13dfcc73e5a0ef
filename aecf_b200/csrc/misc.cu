// Small kernels around the fused pool: column sums (bias gradients), CurriculumMasking.entropy_loss
// forward/backward, and the projection-free single-head attention of the functional fast path.
#include <cmath>

#include "common.cuh"
#include "pool_core.cuh"

namespace aecf {

// ---- column sum ---------------------------------------------------------------------------
// Stage 1: block (32, 8) owns 32 chunks (16 B each) of columns and one split of the rows; the 8 row
// lanes are folded through shared memory in a fixed order.  Stage 2: splits folded in order.
constexpr int COLSUM_ROW_LANES = 8;
constexpr int COLSUM_MAX_SPLITS = 256;

template <typename T>
__global__ void __launch_bounds__(32 * COLSUM_ROW_LANES)
colsum_stage1(const T* __restrict__ x, long long rows, long long cols, long long ld, int splits,
              float* __restrict__ partial) {
    constexpr int V = Vec<T>::N;
    __shared__ float red[COLSUM_ROW_LANES][32 * V + 1];
    const long long chunk = static_cast<long long>(blockIdx.x) * 32 + threadIdx.x;
    const long long col0 = chunk * V;
    const long long per = (rows + splits - 1) / splits;
    const long long r0 = per * blockIdx.y, r1 = min(rows, r0 + per);
    float acc[V];
#pragma unroll
    for (int v = 0; v < V; ++v) acc[v] = 0.f;
    pdl_wait();
    if (col0 < cols) {
        constexpr int U = 8;                               // independent 16-byte loads in flight per thread
        long long r = r0 + threadIdx.y;
        for (; r + (U - 1) * COLSUM_ROW_LANES < r1; r += U * COLSUM_ROW_LANES) {
            uint4 raw[U];
#pragma unroll
            for (int u = 0; u < U; ++u) raw[u] = ldg_stream(x + (r + u * COLSUM_ROW_LANES) * ld + col0);
#pragma unroll
            for (int u = 0; u < U; ++u) {
                float f[V];
                Vec<T>::unpack(raw[u], f);
#pragma unroll
                for (int v = 0; v < V; ++v) acc[v] += f[v];
            }
        }
        for (; r < r1; r += COLSUM_ROW_LANES) {
            float f[V];
            Vec<T>::unpack(ldg_stream(x + r * ld + col0), f);
#pragma unroll
            for (int v = 0; v < V; ++v) acc[v] += f[v];
        }
    }
#pragma unroll
    for (int v = 0; v < V; ++v) red[threadIdx.y][threadIdx.x * V + v] = acc[v];
    __syncthreads();
    if (threadIdx.y == 0 && col0 < cols) {
#pragma unroll
        for (int v = 0; v < V; ++v) {
            float s = 0.f;
#pragma unroll
            for (int y = 0; y < COLSUM_ROW_LANES; ++y) s += red[y][threadIdx.x * V + v];
            partial[static_cast<long long>(blockIdx.y) * cols + col0 + v] = s;
        }
    }
}

template <typename TO>
__global__ void __launch_bounds__(256)
colsum_stage2(const float* __restrict__ partial, long long cols, int splits, TO* __restrict__ out) {
    __shared__ float red[8][33];                       // 32 columns x 8 lanes; fixed-order folds -> deterministic
    const int x = threadIdx.x & 31, y = threadIdx.x >> 5;
    const long long c = static_cast<long long>(blockIdx.x) * 32 + x;
    float s = 0.f;
    pdl_wait();
    if (c < cols) {
#pragma unroll 4
        for (int i = y; i < splits; i += 8) s += partial[static_cast<long long>(i) * cols + c];
    }
    red[y][x] = s;
    __syncthreads();
    if (y != 0 || c >= cols) return;
    s = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) s += red[k][x];
    out[c] = from_float<TO>(s);
}

// ---- parameter shadow -----------------------------------------------------------------------
// fp32 segments -> one bf16 block, round to nearest even (NaN stays NaN, +-inf stays +-inf).  blockIdx.y is the segment;
// blocks stride over its 8-element chunks (two 16-byte loads, one 16-byte store), the last count % 8 elements -- and every
// element of a source that is not 16-byte aligned -- go one at a time.
struct ParamCastParams {
    const float* src[AECF_PARAM_CAST_MAX_SEGMENTS];
    long long count[AECF_PARAM_CAST_MAX_SEGMENTS];
    long long offset[AECF_PARAM_CAST_MAX_SEGMENTS];            // in elements of dst, multiples of 8
    long long chunks[AECF_PARAM_CAST_MAX_SEGMENTS];            // 8-element chunks of the vectorised body (0: src not aligned)
};

__global__ void __launch_bounds__(256)
param_cast_kernel(const ParamCastParams p, __nv_bfloat16* __restrict__ dst) {
    pdl_wait();
    const int seg = blockIdx.y;
    const float* src = p.src[seg];
    const long long n = p.count[seg];
    __nv_bfloat16* out = dst + p.offset[seg];
    const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
    const long long t0 = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    const long long chunks = p.chunks[seg];
    for (long long c = t0; c < chunks; c += stride) {
        const float4 a = *reinterpret_cast<const float4*>(src + 8 * c);
        const float4 b = *reinterpret_cast<const float4*>(src + 8 * c + 4);
        const float f[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
        stg_vec(out + 8 * c, Vec<__nv_bfloat16>::pack(f));
    }
    for (long long i = 8 * chunks + t0; i < n; i += stride) out[i] = from_float<__nv_bfloat16>(src[i]);
}

static int colsum_splits(long long rows) {
    long long s = (rows + 255) / 256;
    if (s < 1) s = 1;
    if (s > COLSUM_MAX_SPLITS) s = COLSUM_MAX_SPLITS;
    return static_cast<int>(s);
}

// ---- entropy loss -------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) entropy_loss_fwd_kernel(const float* __restrict__ e, long long n, float target,
                                                                float* __restrict__ loss) {
    __shared__ float warp_sum[32];
    float acc = 0.f;
    pdl_wait();
    constexpr int U = 8;                                   // independent loads in flight per thread
    for (long long i0 = threadIdx.x; i0 < n; i0 += static_cast<long long>(blockDim.x) * U) {
        float v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const long long i = i0 + static_cast<long long>(u) * blockDim.x;
            v[u] = (i < n) ? e[i] : target;                // out of range: contributes (target - target)^2 = 0
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            bool fin;
            const float d = scrub_entropy(v[u], &fin) - target;
            acc = fmaf(d, d, acc);
        }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(FULL_MASK, acc, off);
    if ((threadIdx.x & 31) == 0) warp_sum[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        float s = 0.f;
        for (int wi = 0; wi < (blockDim.x >> 5); ++wi) s += warp_sum[wi];
        loss[0] = fmaxf(s / static_cast<float>(n), 0.f);              // .mean().clamp_(min=0)
    }
}

__global__ void entropy_loss_bwd_kernel(const float* __restrict__ e, long long n, float target,
                                        const float* __restrict__ d_loss, float* __restrict__ d_e) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    bool fin;
    const float d = scrub_entropy(e[i], &fin) - target;
    d_e[i] = fin ? d_loss[0] * 2.0f * d / static_cast<float>(n) : 0.f;
}


// ---- standalone CurriculumMasking.forward / compute_entropy (reference aecf/AECFLayer.py:101-283) ----
// One thread per row of `len` <= 64 weights; the fused pool kernel carries the same stage for the
// hot path, this one serves direct calls on user-supplied weights (README.md:300-317, 341-350).
constexpr int MASK_MAX_LEN = 64;

__device__ __forceinline__ float entropy_of(const float* w, int len, float log_len, float* raw_out) {
    float acc = 0.f;
    for (int i = 0; i < len; ++i) acc = __fadd_rn(acc, (w[i] == 0.f) ? 0.f : __fmul_rn(w[i], logf(w[i])));
    const float raw = -acc;
    if (raw_out) *raw_out = raw;
    return (raw != raw) ? raw : fminf(fmaxf(raw, 0.f), log_len);
}

__global__ void curriculum_mask_kernel(const float* __restrict__ weights, long long rows, int len, int mode,
                                       float base_mask_prob, int min_active, float log_len, RngKey rng,
                                       float* __restrict__ masked, float* __restrict__ entropy,
                                       float* __restrict__ mask_rate, const float* __restrict__ d_masked = nullptr,
                                       float* __restrict__ d_weights = nullptr) {
    // d_weights != nullptr: the BACKWARD of the training-mode call (mode 1) -- the mask is redrawn from the same Philox
    // row, then d_weights = d(final_weights)/d(weights)^T d_masked; mask, top-k set and entropy carry no gradient
    // (torch.bernoulli / topk indices in the reference, aecf/AECFLayer.py:204-260)
    const long long row = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (row >= rows) return;
    float w[MASK_MAX_LEN];
    for (int i = 0; i < len; ++i) w[i] = weights[row * len + i];
    if (d_weights != nullptr && len <= 1) {                 // a single token passes through unchanged (:159-167)
        for (int i = 0; i < len; ++i) d_weights[row * len + i] = d_masked[row * len + i];
        return;
    }
    if (mode != 1 || len <= 1) {                    // eval mode / entropy only / single token (:150-167)
        const float e = (mode == 1) ? 0.f : entropy_of(w, len, log_len, nullptr);
        if (entropy) entropy[row] = e;
        if (mask_rate) mask_rate[row] = 0.f;
        if (masked) for (int i = 0; i < len; ++i) masked[row * len + i] = w[i];
        return;
    }
    float total = 0.f;
    unsigned long long finite = 0ull;
    for (int i = 0; i < len; ++i) {
        if (fabsf(w[i]) <= 3.402823466e38f) finite |= 1ull << i;
        else w[i] = 0.f;
        total = __fadd_rn(total, w[i]);
    }
    const bool degenerate = total < 1e-8f;
    const float uniform = static_cast<float>(1.0 / static_cast<double>(len));
    for (int i = 0; i < len; ++i) w[i] = degenerate ? uniform : w[i] / total;
    const float e = entropy_of(w, len, log_len, nullptr);
    const float norm_entropy = fminf(fmaxf(e / log_len, 0.f), 1.f);
    const float keep_prob = fminf(fmaxf(__fsub_rn(1.0f, __fmul_rn(base_mask_prob, norm_entropy)), 0.f), 1.f);
    unsigned long long bits = 0ull;
    int active = 0;
    for (int blk = 0; blk < (len + 3) / 4; ++blk) {
        float u[4];
        draw4(rng, static_cast<unsigned long long>(row), STREAM_MASK, 0u, blk, u);
        for (int i = 0; i < 4; ++i) {
            const int m = 4 * blk + i;
            if (m < len && u[i] <= keep_prob) { bits |= 1ull << m; ++active; }
        }
    }
    const int need = min(min_active, len);
    if (active < need) {
        bits = 0ull;
        for (int i = 0; i < len; ++i) {
            int rank = 0;
            for (int j = 0; j < len; ++j) rank += (w[j] > w[i] || (w[j] == w[i] && j < i)) ? 1 : 0;
            if (rank < need) bits |= 1ull << i;
        }
        active = need;
    }
    float kept_sum = 0.f;
    for (int i = 0; i < len; ++i) kept_sum = __fadd_rn(kept_sum, ((bits >> i) & 1ull) ? w[i] : 0.f);
    const bool valid = kept_sum > 1e-8f;
    if (d_weights != nullptr) {
        // valid: final = wn m / kept_sum (degree 0 in wn, so the 1/total of wn = w / total is all that is left of it);
        // fallback: final = wn.  A degenerate row (wn = uniform) and non-finite entries get no gradient.
        float dot = 0.f;
        for (int i = 0; i < len; ++i) {
            const float fin = valid ? ((((bits >> i) & 1ull) ? w[i] : 0.f) / kept_sum) : w[i];
            dot = fmaf(d_masked[row * len + i], fin, dot);
        }
        for (int i = 0; i < len; ++i) {
            float d = 0.f;
            if (!degenerate && ((finite >> i) & 1ull)) {
                const float g = d_masked[row * len + i];
                d = valid ? (((bits >> i) & 1ull) ? (g - dot) / kept_sum / total : 0.f) : (g - dot) / total;
            }
            d_weights[row * len + i] = d;
        }
        return;
    }
    if (masked)
        for (int i = 0; i < len; ++i)
            masked[row * len + i] = valid ? (((bits >> i) & 1ull) ? w[i] : 0.f) / kept_sum : w[i];
    if (entropy) entropy[row] = e;
    if (mask_rate) mask_rate[row] = __fsub_rn(1.0f, static_cast<float>(active) / static_cast<float>(len));
}

// Eval-mode entropy stays attached (:151-156).  d_weights[i] = -g (xlogy(w_i != 0, w_i) + w_i / w_i) with g = d_entropy
// inside the clamp, else 0: autograd's backward of clamp(-sum xlogy(w, w)) term by term, so that a zero weight gets
// 0 / 0 = NaN as it does in torch -- also where the clamp passes no gradient -- and not -(log 0 + 1) = +inf.
__global__ void entropy_bwd_kernel(const float* __restrict__ weights, long long rows, int len, float log_len,
                                   const float* __restrict__ d_entropy, float* __restrict__ d_weights) {
    const long long row = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (row >= rows) return;
    float w[MASK_MAX_LEN];
    for (int i = 0; i < len; ++i) w[i] = weights[row * len + i];
    float raw;
    entropy_of(w, len, log_len, &raw);
    const bool inside = (raw >= 0.f) && (raw <= log_len);
    const float g = inside ? d_entropy[row] : 0.f;
    for (int i = 0; i < len; ++i)
        d_weights[row * len + i] = -((w[i] != 0.f ? logf(w[i]) : 0.f) + w[i] / w[i]) * g;
}

// ---- projection-free single-head attention (reference aecf/AECFLayer.py:556-581) ------------
// One warp per query row, online softmax over the source tokens, any src_len.
template <typename T, int JMAX>
__global__ void __launch_bounds__(256) sdpa_fwd_kernel(const T* __restrict__ q, const T* __restrict__ k,
                                                       const T* __restrict__ v, T* __restrict__ out, long long rows,
                                                       int tgt_len, int src_len, int D, float scale) {
    constexpr int V = Vec<T>::N;
    const int lane = threadIdx.x & 31;
    const long long qrow = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (qrow >= rows) return;
    const long long b = qrow / tgt_len;
    const int NC = D / V;
    float qf[JMAX][V], acc[JMAX][V];
#pragma unroll
    for (int j = 0; j < JMAX; ++j) {
        const int c = lane + 32 * j;
#pragma unroll
        for (int x = 0; x < V; ++x) { qf[j][x] = 0.f; acc[j][x] = 0.f; }
        if (c < NC) Vec<T>::unpack(ldg_stream(q + qrow * D + static_cast<long long>(c) * V), qf[j]);
    }
    float run_max = -INFINITY, run_sum = 0.f;
    for (int t = 0; t < src_len; ++t) {
        const long long krow = (b * src_len + t) * D;
        float dot = 0.f;
#pragma unroll
        for (int j = 0; j < JMAX; ++j) {
            const int c = lane + 32 * j;
            if (c < NC) {
                float f[V];
                Vec<T>::unpack(ldg_stream(k + krow + static_cast<long long>(c) * V), f);
#pragma unroll
                for (int x = 0; x < V; ++x) dot = fmaf(qf[j][x], f[x], dot);
            }
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) dot += __shfl_xor_sync(FULL_MASK, dot, off);
        const float s = dot * scale;                                   // bmm(q, k^T) * scale (:577)
        const float new_max = fmaxf(run_max, s);
        const float corr = expf(run_max - new_max), pexp = expf(s - new_max);
        run_sum = run_sum * corr + pexp;
        run_max = new_max;
#pragma unroll
        for (int j = 0; j < JMAX; ++j) {
            const int c = lane + 32 * j;
            if (c < NC) {
                float f[V];
                Vec<T>::unpack(ldg_stream(v + krow + static_cast<long long>(c) * V), f);
#pragma unroll
                for (int x = 0; x < V; ++x) acc[j][x] = fmaf(pexp, f[x], acc[j][x] * corr);
            }
        }
    }
#pragma unroll
    for (int j = 0; j < JMAX; ++j) {
        const int c = lane + 32 * j;
        if (c < NC) {
#pragma unroll
            for (int x = 0; x < V; ++x) acc[j][x] = acc[j][x] / run_sum;
            stg_vec(out + qrow * D + static_cast<long long>(c) * V, Vec<T>::pack(acc[j]));
        }
    }
}

template <typename T>
static int launch_sdpa(const void* q, const void* k, const void* v, void* out, long long rows, int tgt, int src,
                       int D, cudaStream_t s) {
    constexpr int V = Vec<T>::N;
    const int NC = D / V;
    const float scale = static_cast<float>(1.0 / std::sqrt(static_cast<double>(D)));   // query.size(-1) ** -0.5 (:574)
    const unsigned grid = static_cast<unsigned>((rows + 7) / 8);
#define AECF_SDPA(JM)                                                                                        \
    AECF_CUDA_OK(launch_plain(sdpa_fwd_kernel<T, JM>, dim3(grid), dim3(256), 0, s, static_cast<const T*>(q),   \
                              static_cast<const T*>(k), static_cast<const T*>(v), static_cast<T*>(out), rows, tgt, src, D, scale))
    if (NC <= 32) AECF_SDPA(1);
    else if (NC <= 64) AECF_SDPA(2);
    else if (NC <= 128) AECF_SDPA(4);
    else if (NC <= 256) AECF_SDPA(8);
    else return AECF_ERR_UNSUPPORTED;
#undef AECF_SDPA
    count_launch();
    return AECF_OK;
}


// ---- backward of the projection-free attention (reference aecf/AECFLayer.py:573-581 is differentiable) -----------------
// out[s] = sum_t p[s,t] v[t],  p = softmax_t(scale q[s] . k[t]):
//   dP[s,t] = g[s] . v[t]      delta[s] = sum_t p dP      dS = p (dP - delta)
//   dq[s] = scale sum_t dS k[t]        dk[t] = scale sum_s dS q[s]        dv[t] = sum_s p g[s]
// Two kernels, nothing stored by the forward: one warp per QUERY row recomputes its scores (log-sum-exp, then delta, then
// dq: three passes over the sample's keys, which sit in L1/L2) and leaves lse / delta; one warp per KEY row then walks the
// sample's queries.  A warp covers the row chunk-wise (16 bytes per lane) and dots are xor-shuffle reductions.
template <typename T, int JMAX>
__device__ __forceinline__ float sdpa_dot(const float (&a)[JMAX][Vec<T>::N], const T* row, int lane, int NC) {
    constexpr int V = Vec<T>::N;
    float dot = 0.f;
#pragma unroll
    for (int j = 0; j < JMAX; ++j) {
        const int c = lane + 32 * j;
        if (c < NC) {
            float f[V];
            Vec<T>::unpack(ldg_cached(row + static_cast<long long>(c) * V), f);
#pragma unroll
            for (int x = 0; x < V; ++x) dot = fmaf(a[j][x], f[x], dot);
        }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) dot += __shfl_xor_sync(FULL_MASK, dot, off);
    return dot;
}

template <typename T, int JMAX>
__device__ __forceinline__ void sdpa_load(float (&a)[JMAX][Vec<T>::N], const T* row, int lane, int NC) {
    constexpr int V = Vec<T>::N;
#pragma unroll
    for (int j = 0; j < JMAX; ++j) {
        const int c = lane + 32 * j;
#pragma unroll
        for (int x = 0; x < V; ++x) a[j][x] = 0.f;
        if (c < NC) Vec<T>::unpack(ldg_cached(row + static_cast<long long>(c) * V), a[j]);
    }
}

template <typename T, int JMAX>
__global__ void __launch_bounds__(256) sdpa_bwd_q_kernel(const T* __restrict__ q, const T* __restrict__ k, const T* __restrict__ v,
                                                         const T* __restrict__ g, T* __restrict__ d_q, float* __restrict__ lse,
                                                         float* __restrict__ delta, long long rows, int tgt_len, int src_len,
                                                         int D, float scale) {
    constexpr int V = Vec<T>::N;
    const int lane = threadIdx.x & 31;
    const long long qrow = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (qrow >= rows) return;
    const long long b = qrow / tgt_len;
    const int NC = D / V;
    float qf[JMAX][V], gf[JMAX][V], acc[JMAX][V];
    sdpa_load<T, JMAX>(qf, q + qrow * D, lane, NC);
    sdpa_load<T, JMAX>(gf, g + qrow * D, lane, NC);
    float mx = -INFINITY, sum = 0.f;
    for (int t = 0; t < src_len; ++t) {
        const float s = sdpa_dot<T, JMAX>(qf, k + (b * src_len + t) * D, lane, NC) * scale;
        const float nm = fmaxf(mx, s);
        sum = sum * expf(mx - nm) + expf(s - nm);
        mx = nm;
    }
    const float l = mx + logf(sum);
    float dl = 0.f;
    for (int t = 0; t < src_len; ++t) {
        const long long krow = (b * src_len + t) * D;
        const float p = expf(sdpa_dot<T, JMAX>(qf, k + krow, lane, NC) * scale - l);
        dl = fmaf(p, sdpa_dot<T, JMAX>(gf, v + krow, lane, NC), dl);
    }
#pragma unroll
    for (int j = 0; j < JMAX; ++j)
#pragma unroll
        for (int x = 0; x < V; ++x) acc[j][x] = 0.f;
    for (int t = 0; t < src_len; ++t) {
        const long long krow = (b * src_len + t) * D;
        const float p = expf(sdpa_dot<T, JMAX>(qf, k + krow, lane, NC) * scale - l);
        const float ds = p * (sdpa_dot<T, JMAX>(gf, v + krow, lane, NC) - dl) * scale;
#pragma unroll
        for (int j = 0; j < JMAX; ++j) {
            const int c = lane + 32 * j;
            if (c < NC) {
                float f[V];
                Vec<T>::unpack(ldg_cached(k + krow + static_cast<long long>(c) * V), f);
#pragma unroll
                for (int x = 0; x < V; ++x) acc[j][x] = fmaf(ds, f[x], acc[j][x]);
            }
        }
    }
#pragma unroll
    for (int j = 0; j < JMAX; ++j) {
        const int c = lane + 32 * j;
        if (c < NC) stg_vec(d_q + qrow * D + static_cast<long long>(c) * V, Vec<T>::pack(acc[j]));
    }
    if (lane == 0) { lse[qrow] = l; delta[qrow] = dl; }
}

template <typename T, int JMAX>
__global__ void __launch_bounds__(256) sdpa_bwd_kv_kernel(const T* __restrict__ q, const T* __restrict__ k, const T* __restrict__ v,
                                                          const T* __restrict__ g, const float* __restrict__ lse,
                                                          const float* __restrict__ delta, T* __restrict__ d_k, T* __restrict__ d_v,
                                                          long long key_rows, int tgt_len, int src_len, int D, float scale) {
    constexpr int V = Vec<T>::N;
    const int lane = threadIdx.x & 31;
    const long long krow = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (krow >= key_rows) return;
    const long long b = krow / src_len;
    const int NC = D / V;
    float kf[JMAX][V], vf[JMAX][V], dk[JMAX][V], dv[JMAX][V];
    sdpa_load<T, JMAX>(kf, k + krow * D, lane, NC);
    sdpa_load<T, JMAX>(vf, v + krow * D, lane, NC);
#pragma unroll
    for (int j = 0; j < JMAX; ++j)
#pragma unroll
        for (int x = 0; x < V; ++x) { dk[j][x] = 0.f; dv[j][x] = 0.f; }
    for (int s = 0; s < tgt_len; ++s) {
        const long long qrow = b * tgt_len + s;
        const float p = expf(sdpa_dot<T, JMAX>(kf, q + qrow * D, lane, NC) * scale - lse[qrow]);
        const float ds = p * (sdpa_dot<T, JMAX>(vf, g + qrow * D, lane, NC) - delta[qrow]) * scale;
#pragma unroll
        for (int j = 0; j < JMAX; ++j) {
            const int c = lane + 32 * j;
            if (c < NC) {
                float fq[V], fg[V];
                Vec<T>::unpack(ldg_cached(q + qrow * D + static_cast<long long>(c) * V), fq);
                Vec<T>::unpack(ldg_cached(g + qrow * D + static_cast<long long>(c) * V), fg);
#pragma unroll
                for (int x = 0; x < V; ++x) { dk[j][x] = fmaf(ds, fq[x], dk[j][x]); dv[j][x] = fmaf(p, fg[x], dv[j][x]); }
            }
        }
    }
#pragma unroll
    for (int j = 0; j < JMAX; ++j) {
        const int c = lane + 32 * j;
        if (c < NC) {
            stg_vec(d_k + krow * D + static_cast<long long>(c) * V, Vec<T>::pack(dk[j]));
            stg_vec(d_v + krow * D + static_cast<long long>(c) * V, Vec<T>::pack(dv[j]));
        }
    }
}

template <typename T>
static int launch_sdpa_bwd(const void* q, const void* k, const void* v, const void* g, void* d_q, void* d_k, void* d_v,
                           float* ws, long long batch, int tgt, int src, int D, cudaStream_t s) {
    constexpr int V = Vec<T>::N;
    const int NC = D / V;
    const float scale = static_cast<float>(1.0 / std::sqrt(static_cast<double>(D)));
    const long long qrows = batch * tgt, krows = batch * src;
    float* lse = ws;
    float* delta = ws + qrows;
#define AECF_SDPA_BWD(JM)                                                                                              \
    do {                                                                                                               \
        AECF_CUDA_OK(launch_plain(sdpa_bwd_q_kernel<T, JM>, dim3(static_cast<unsigned>((qrows + 7) / 8)), dim3(256), 0, s,         \
                                  static_cast<const T*>(q), static_cast<const T*>(k), static_cast<const T*>(v),        \
                                  static_cast<const T*>(g), static_cast<T*>(d_q), lse, delta, qrows, tgt, src, D, scale));          \
        AECF_CUDA_OK(launch_plain(sdpa_bwd_kv_kernel<T, JM>, dim3(static_cast<unsigned>((krows + 7) / 8)), dim3(256), 0, s,        \
                                  static_cast<const T*>(q), static_cast<const T*>(k), static_cast<const T*>(v),        \
                                  static_cast<const T*>(g), static_cast<const float*>(lse), static_cast<const float*>(delta),      \
                                  static_cast<T*>(d_k), static_cast<T*>(d_v), krows, tgt, src, D, scale));                         \
    } while (0)
    if (NC <= 32) AECF_SDPA_BWD(1);
    else if (NC <= 64) AECF_SDPA_BWD(2);
    else if (NC <= 128) AECF_SDPA_BWD(4);
    else if (NC <= 256) AECF_SDPA_BWD(8);
    else return AECF_ERR_UNSUPPORTED;
#undef AECF_SDPA_BWD
    count_launch(2);
    return AECF_OK;
}

}  // namespace aecf

using namespace aecf;

extern "C" {

size_t aecf_colsum_workspace_bytes(int64_t rows, int64_t cols) {
    if (rows < 0 || cols <= 0) return 0;
    return static_cast<size_t>(colsum_splits(rows)) * static_cast<size_t>(cols) * sizeof(float);
}

int aecf_colsum(int32_t device, int32_t dtype_x, int32_t dtype_out, const void* x, int64_t rows, int64_t cols,
                int64_t ld, void* out, void* workspace, size_t workspace_bytes, void* stream) {
    if (!x || !out || !workspace || rows < 0 || cols <= 0 || ld < cols) return AECF_ERR_INVALID;
    if ((dtype_x != AECF_F32 && dtype_x != AECF_BF16) || (dtype_out != AECF_F32 && dtype_out != AECF_BF16))
        return AECF_ERR_INVALID;
    const int V = dtype_x == AECF_BF16 ? 8 : 4;
    const size_t es = dtype_x == AECF_BF16 ? 2 : 4;
    if (cols % V != 0) return AECF_ERR_UNSUPPORTED;
    if (!aligned16(x) || (static_cast<size_t>(ld) * es) % 16 != 0) return AECF_ERR_ALIGNMENT;
    if (workspace_bytes < aecf_colsum_workspace_bytes(rows, cols)) return AECF_ERR_WORKSPACE;
    DeviceScope device_scope__(device);
    int rc = device_scope__.rc;
    if (rc != AECF_OK) return rc;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    TimedLaunch timed(s);
    const int splits = colsum_splits(rows);
    const dim3 block(32, COLSUM_ROW_LANES), grid(static_cast<unsigned>((cols / V + 31) / 32), splits);
    float* partial = static_cast<float*>(workspace);
    if (dtype_x == AECF_BF16)
        AECF_CUDA_OK(launch_pdl(colsum_stage1<__nv_bfloat16>, grid, block, 0, s, static_cast<const __nv_bfloat16*>(x), rows, cols,
                                ld, splits, partial));
    else
        AECF_CUDA_OK(launch_pdl(colsum_stage1<float>, grid, block, 0, s, static_cast<const float*>(x), rows, cols, ld, splits,
                                partial));
    const dim3 g2(static_cast<unsigned>((cols + 31) / 32));
    if (dtype_out == AECF_BF16)
        AECF_CUDA_OK(launch_pdl(colsum_stage2<__nv_bfloat16>, g2, dim3(256), 0, s, partial, cols, splits,
                                static_cast<__nv_bfloat16*>(out)));
    else
        AECF_CUDA_OK(launch_pdl(colsum_stage2<float>, g2, dim3(256), 0, s, partial, cols, splits, static_cast<float*>(out)));
    count_launch(2);
    return AECF_OK;
}

int aecf_param_cast(int32_t device, int32_t segments, const float* const* src, const int64_t* counts, void* dst,
                    void* stream) {
    if (!src || !counts || !dst || segments <= 0 || segments > AECF_PARAM_CAST_MAX_SEGMENTS) return AECF_ERR_INVALID;
    if (!aligned16(dst)) return AECF_ERR_ALIGNMENT;
    ParamCastParams p{};
    long long offset = 0, widest = 0;
    for (int i = 0; i < segments; ++i) {
        if (counts[i] < 0 || (counts[i] > 0 && !src[i])) return AECF_ERR_INVALID;
        p.src[i] = src[i]; p.count[i] = counts[i]; p.offset[i] = offset;
        p.chunks[i] = aligned16(src[i]) ? counts[i] / 8 : 0;
        offset += (counts[i] + 7) / 8 * 8;                     // the next segment starts on a 16-byte boundary
        widest = counts[i] > widest ? counts[i] : widest;
    }
    if (widest == 0) return AECF_OK;
    DeviceScope device_scope__(device);
    int rc = device_scope__.rc;
    if (rc != AECF_OK) return rc;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    TimedLaunch timed(s, AECF_SITE_PARAM_CAST);
    const long long blocks = (widest + 8 * 256 - 1) / (8 * 256);
    const dim3 grid(static_cast<unsigned>(blocks < 1024 ? blocks : 1024), static_cast<unsigned>(segments));
    AECF_CUDA_OK(launch_pdl(param_cast_kernel, grid, dim3(256), 0, s, p, static_cast<__nv_bfloat16*>(dst)));
    count_launch();
    return AECF_OK;
}

int aecf_entropy_loss_fwd(int32_t device, const float* entropy, int64_t n, float target, float* loss, void* stream) {
    if (!entropy || !loss || n <= 0) return AECF_ERR_INVALID;
    DeviceScope device_scope__(device);
    int rc = device_scope__.rc;
    if (rc != AECF_OK) return rc;
    TimedLaunch timed(static_cast<cudaStream_t>(stream), AECF_SITE_ENTROPY_LOSS);
    AECF_CUDA_OK(launch_pdl(entropy_loss_fwd_kernel, dim3(1), dim3(1024), 0, static_cast<cudaStream_t>(stream), entropy,
                            static_cast<long long>(n), target, loss));
    count_launch();
    return AECF_OK;
}

int aecf_entropy_loss_bwd(int32_t device, const float* entropy, int64_t n, float target, const float* d_loss,
                          float* d_entropy, void* stream) {
    if (!entropy || !d_loss || !d_entropy || n <= 0) return AECF_ERR_INVALID;
    DeviceScope device_scope__(device);
    int rc = device_scope__.rc;
    if (rc != AECF_OK) return rc;
    AECF_CUDA_OK(launch_plain(entropy_loss_bwd_kernel, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0,
                              static_cast<cudaStream_t>(stream), entropy, static_cast<long long>(n), target, d_loss, d_entropy));
    count_launch();
    return AECF_OK;
}

int aecf_curriculum_mask(int32_t device, const float* weights, int64_t rows, int32_t len, int32_t mode,
                         float base_mask_prob, int32_t min_active, uint64_t seed, uint64_t offset, uint64_t row0,
                         float* masked, float* entropy, float* mask_rate, void* stream) {
    if (!weights || rows < 0 || len <= 0 || mode < 1 || mode > 3 || (offset >> 32)) return AECF_ERR_INVALID;
    if (len > MASK_MAX_LEN) return AECF_ERR_UNSUPPORTED;
    if (rows == 0) return AECF_OK;
    DeviceScope device_scope__(device);
    int rc = device_scope__.rc;
    if (rc != AECF_OK) return rc;
    RngKey rng;
    rng.k0 = static_cast<uint32_t>(seed); rng.k1 = static_cast<uint32_t>(seed >> 32);
    rng.offset = static_cast<uint32_t>(offset); rng.row0 = row0;
    const float log_len = static_cast<float>(std::log(static_cast<double>(len)));
    AECF_CUDA_OK(launch_plain(curriculum_mask_kernel, dim3(static_cast<unsigned>((rows + 127) / 128)), dim3(128), 0,
                              static_cast<cudaStream_t>(stream), weights, static_cast<long long>(rows), len, mode, base_mask_prob,
                              min_active, log_len, rng, masked, entropy, mask_rate, static_cast<const float*>(nullptr),
                              static_cast<float*>(nullptr)));
    count_launch();
    return AECF_OK;
}

int aecf_curriculum_mask_bwd(int32_t device, const float* weights, int64_t rows, int32_t len, float base_mask_prob,
                             int32_t min_active, uint64_t seed, uint64_t offset, uint64_t row0, const float* d_masked,
                             float* d_weights, void* stream) {
    if (!weights || !d_masked || !d_weights || rows < 0 || len <= 0 || (offset >> 32)) return AECF_ERR_INVALID;
    if (len > MASK_MAX_LEN) return AECF_ERR_UNSUPPORTED;
    if (rows == 0) return AECF_OK;
    DeviceScope device_scope__(device);
    int rc = device_scope__.rc;
    if (rc != AECF_OK) return rc;
    RngKey rng;
    rng.k0 = static_cast<uint32_t>(seed); rng.k1 = static_cast<uint32_t>(seed >> 32);
    rng.offset = static_cast<uint32_t>(offset); rng.row0 = row0;
    const float log_len = static_cast<float>(std::log(static_cast<double>(len)));
    AECF_CUDA_OK(launch_plain(curriculum_mask_kernel, dim3(static_cast<unsigned>((rows + 127) / 128)), dim3(128), 0,
                              static_cast<cudaStream_t>(stream), weights, static_cast<long long>(rows), len, 1, base_mask_prob,
                              min_active, log_len, rng, static_cast<float*>(nullptr), static_cast<float*>(nullptr),
                              static_cast<float*>(nullptr), d_masked, d_weights));
    count_launch();
    return AECF_OK;
}

int aecf_entropy_bwd(int32_t device, const float* weights, int64_t rows, int32_t len, const float* d_entropy,
                     float* d_weights, void* stream) {
    if (!weights || !d_entropy || !d_weights || rows < 0 || len <= 0) return AECF_ERR_INVALID;
    if (len > MASK_MAX_LEN) return AECF_ERR_UNSUPPORTED;
    if (rows == 0) return AECF_OK;
    DeviceScope device_scope__(device);
    int rc = device_scope__.rc;
    if (rc != AECF_OK) return rc;
    const float log_len = static_cast<float>(std::log(static_cast<double>(len)));
    AECF_CUDA_OK(launch_plain(entropy_bwd_kernel, dim3(static_cast<unsigned>((rows + 127) / 128)), dim3(128), 0,
                              static_cast<cudaStream_t>(stream), weights, static_cast<long long>(rows), len, log_len, d_entropy,
                              d_weights));
    count_launch();
    return AECF_OK;
}

int aecf_sdpa_fwd(int32_t device, int32_t dtype, const void* q, const void* k, const void* v, void* out,
                  int64_t batch, int32_t tgt_len, int32_t src_len, int32_t embed_dim, void* stream) {
    if (!q || !k || !v || !out || batch < 0 || tgt_len <= 0 || src_len <= 0 || embed_dim <= 0) return AECF_ERR_INVALID;
    if (dtype != AECF_F32 && dtype != AECF_BF16) return AECF_ERR_INVALID;
    if (batch == 0) return AECF_OK;
    const int V = dtype == AECF_BF16 ? 8 : 4;
    if (embed_dim % V != 0) return AECF_ERR_UNSUPPORTED;
    if (!aligned16(q) || !aligned16(k) || !aligned16(v) || !aligned16(out)) return AECF_ERR_ALIGNMENT;
    DeviceScope device_scope__(device);
    int rc = device_scope__.rc;
    if (rc != AECF_OK) return rc;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const long long rows = static_cast<long long>(batch) * tgt_len;
    return dtype == AECF_BF16 ? launch_sdpa<__nv_bfloat16>(q, k, v, out, rows, tgt_len, src_len, embed_dim, s)
                              : launch_sdpa<float>(q, k, v, out, rows, tgt_len, src_len, embed_dim, s);
}

/* d_q / d_k / d_v of aecf_sdpa_fwd for an upstream gradient d_out [B, tgt, D]; workspace >= 2 * B * tgt_len floats */
int aecf_sdpa_bwd(int32_t device, int32_t dtype, const void* q, const void* k, const void* v, const void* d_out, void* d_q,
                  void* d_k, void* d_v, void* workspace, size_t workspace_bytes, int64_t batch, int32_t tgt_len,
                  int32_t src_len, int32_t embed_dim, void* stream) {
    if (!q || !k || !v || !d_out || !d_q || !d_k || !d_v || !workspace || batch < 0 || tgt_len <= 0 || src_len <= 0 || embed_dim <= 0)
        return AECF_ERR_INVALID;
    if (dtype != AECF_F32 && dtype != AECF_BF16) return AECF_ERR_INVALID;
    if (batch == 0) return AECF_OK;
    const int V = dtype == AECF_BF16 ? 8 : 4;
    if (embed_dim % V != 0) return AECF_ERR_UNSUPPORTED;
    if (!aligned16(q) || !aligned16(k) || !aligned16(v) || !aligned16(d_out) || !aligned16(d_q) || !aligned16(d_k) || !aligned16(d_v))
        return AECF_ERR_ALIGNMENT;
    if (workspace_bytes < static_cast<size_t>(2) * batch * tgt_len * sizeof(float)) return AECF_ERR_WORKSPACE;
    DeviceScope device_scope__(device);
    int rc = device_scope__.rc;
    if (rc != AECF_OK) return rc;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    return dtype == AECF_BF16
        ? launch_sdpa_bwd<__nv_bfloat16>(q, k, v, d_out, d_q, d_k, d_v, static_cast<float*>(workspace), batch, tgt_len, src_len, embed_dim, s)
        : launch_sdpa_bwd<float>(q, k, v, d_out, d_q, d_k, d_v, static_cast<float*>(workspace), batch, tgt_len, src_len, embed_dim, s);
}

}  // extern "C"
