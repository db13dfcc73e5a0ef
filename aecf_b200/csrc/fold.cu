// Folded key projection: the two small kernels either side of the GEMMs (include/aecf_b200.h, "folded key
// projection").  With one fusion query for all rows (reference aecf/AECFLayer.py:694 expands a [1,1,D]
// parameter) the key projection of torch/nn/functional.py:5855 collapses to one D-vector per head:
//     score[b,h,m] = scale * q_h . (Wk_h x[b,m] + bk_h) = x[b,m] . Qk[h] + const(h)
// so K is never materialised, forward or backward.
#include "common.cuh"

namespace aecf {

// folded_w = [ Wv (D rows) ; Qk (H rows) ; zeros (HSP - H rows) ], each row D wide.
//   blocks [0, fold_blocks): block (strip of 32 columns d, row r < HSP), 32 x 8 threads: the 8 thread rows split the
//       head_dim terms of  Qk[r, d] = scale * sum_j q[r*hd + j] * Wk[r*hd + j, d]  (every load independent) and are
//       folded through shared memory in a fixed order
//   the remaining blocks copy Wv, 16 bytes per thread, grid-stride.
template <typename T>
__global__ void __launch_bounds__(256)
fold_prepare_kernel(const float* __restrict__ q_proj, const T* __restrict__ in_proj_weight, int D, int H, int HSP,
                    float scale, int fold_blocks, T* __restrict__ folded_w) {
    __shared__ float red[8][33];
    pdl_wait();
    const int hd = D / H;
    if (static_cast<int>(blockIdx.x) < fold_blocks) {
        const int strips = (D + 31) / 32;
        const int r = blockIdx.x / strips;
        const int x = threadIdx.x & 31, y = threadIdx.x >> 5;
        const int d = (blockIdx.x - r * strips) * 32 + x;
        float acc = 0.f;
        if (r < H && d < D) {
            const T* wk = in_proj_weight + (static_cast<size_t>(D) + static_cast<size_t>(r) * hd) * D + d;
            const float* q = q_proj + r * hd;
#pragma unroll 4
            for (int j = y; j < hd; j += 8) acc = fmaf(__ldg(q + j), to_float<T>(wk[static_cast<size_t>(j) * D]), acc);
        }
        red[y][x] = acc;
        __syncthreads();
        if (y != 0 || d >= D) return;
        float s = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) s += red[k][x];
        folded_w[(static_cast<size_t>(D) + r) * D + d] = from_float<T>(s * scale);
        return;
    }
    const uint4* src = reinterpret_cast<const uint4*>(in_proj_weight + 2 * static_cast<size_t>(D) * D);
    uint4* dst = reinterpret_cast<uint4*>(folded_w);
    const size_t n16 = static_cast<size_t>(D) * D * sizeof(T) / 16;
    const size_t stride = static_cast<size_t>(gridDim.x - fold_blocks) * 256;
    for (size_t i = static_cast<size_t>(blockIdx.x - fold_blocks) * 256 + threadIdx.x; i < n16; i += stride) dst[i] = src[i];
}

// The same, starting from the UNPROJECTED fusion query: q_proj = Wq q0 + bq (torch/nn/functional.py:5854) is computed here,
// so the forward of a shared query pays one launch before its GEMM instead of two (GEMV, then the fold).  Every block of
// head r first forms that head's head_dim entries of q_proj in shared memory (one warp per entry, lanes along D, fixed
// xor-shuffle order; 16 blocks repeat the same 64 dots of a 512-vector -- cheaper than a launch boundary); the block of
// strip 0 also writes them out, the backward needs q_proj.
template <typename T>
__global__ void __launch_bounds__(256, 1)
fold_prepare_query_kernel(const T* __restrict__ query, const T* __restrict__ in_proj_weight, const T* __restrict__ in_proj_bias,
                          int D, int H, int HSP, float scale, int fold_blocks, float* __restrict__ q_proj,
                          T* __restrict__ folded_w) {
    __shared__ float red[8][33];
    AECF_DYNAMIC_SMEM(float, qh);                                 // [head_dim]
    pdl_wait();
    const int hd = D / H;
    if (static_cast<int>(blockIdx.x) < fold_blocks) {
        const int strips = (D + 31) / 32;
        const int r = blockIdx.x / strips;
        const int strip = blockIdx.x - r * strips;
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
        if (r < H) {
            // 16-byte loads, every load of a dot in flight before the first multiply; lanes cover the row chunk-wise and
            // are folded by xor shuffles; chunks in order, so the value does not depend on the block that computes it
            constexpr int V = Vec<T>::N;
            const int NC = D / V;
            // eight dots (rows j, j + 8, ... of the head) and their biases share one trip to memory
            constexpr int Q = 8;
            for (int j0 = warp; j0 < hd; j0 += 8 * Q) {
                float acc[Q], bq[Q];
#pragma unroll
                for (int q = 0; q < Q; ++q) {
                    acc[q] = 0.f;
                    const int j = j0 + 8 * q;
                    bq[q] = (in_proj_bias != nullptr && j < hd) ? to_float<T>(in_proj_bias[r * hd + j]) : 0.f;
                }
                for (int c0 = lane; c0 < NC; c0 += 64) {
                    uint4 a[2], b[Q][2];
#pragma unroll
                    for (int u = 0; u < 2; ++u) {
                        const int c = c0 + 32 * u;
                        a[u] = c < NC ? ldg_cached(query + static_cast<size_t>(c) * V) : make_uint4(0, 0, 0, 0);
#pragma unroll
                        for (int q = 0; q < Q; ++q) {
                            const int j = j0 + 8 * q;
                            b[q][u] = (c < NC && j < hd) ? ldg_cached(in_proj_weight + static_cast<size_t>(r * hd + j) * D + static_cast<size_t>(c) * V)
                                                         : make_uint4(0, 0, 0, 0);
                        }
                    }
#pragma unroll
                    for (int u = 0; u < 2; ++u) {
                        float fa[V];
                        Vec<T>::unpack(a[u], fa);
#pragma unroll
                        for (int q = 0; q < Q; ++q) {
                            float fb[V];
                            Vec<T>::unpack(b[q][u], fb);
#pragma unroll
                            for (int v = 0; v < V; ++v) acc[q] = fmaf(fa[v], fb[v], acc[q]);
                        }
                    }
                }
#pragma unroll
                for (int q = 0; q < Q; ++q) {
                    const int j = j0 + 8 * q;
                    float s = acc[q];
#pragma unroll
                    for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(FULL_MASK, s, off);
                    if (j < hd) {
                        s += bq[q];
                        if (lane == 0) {
                            qh[j] = s;
                            if (strip == 0) q_proj[r * hd + j] = s;
                        }
                    }
                }
            }
        }
        __syncthreads();
        const int x = threadIdx.x & 31, y = threadIdx.x >> 5;
        const int d = strip * 32 + x;
        float acc = 0.f;
        if (r < H && d < D) {
            const T* wk = in_proj_weight + (static_cast<size_t>(D) + static_cast<size_t>(r) * hd) * D + d;
#pragma unroll 8
            for (int j = y; j < hd; j += 8) acc = fmaf(qh[j], to_float<T>(wk[static_cast<size_t>(j) * D]), acc);
        }
        red[y][x] = acc;
        __syncthreads();
        if (y != 0 || d >= D) return;
        float s = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) s += red[k][x];
        folded_w[(static_cast<size_t>(D) + r) * D + d] = from_float<T>(s * scale);
        return;
    }
    const uint4* src = reinterpret_cast<const uint4*>(in_proj_weight + 2 * static_cast<size_t>(D) * D);
    uint4* dst = reinterpret_cast<uint4*>(folded_w);
    const size_t n16 = static_cast<size_t>(D) * D * sizeof(T) / 16;
    const size_t stride = static_cast<size_t>(gridDim.x - fold_blocks) * 256;
    for (size_t i = static_cast<size_t>(blockIdx.x - fold_blocks) * 256 + threadIdx.x; i < n16; i += stride) dst[i] = src[i];
}

// g = [dWv (D rows) ; R (H rows) ; ...] fp32, each row D wide; one warp per in-projection row i (head h = i / hd):
//   dWv[i, :] = g[i, :]              dWk[i, :] = scale * q[i] * R[h, :]        d_q[i] = scale * Wk[i, :] . R[h, :]
template <typename T>
__global__ void __launch_bounds__(256)
fold_finish_kernel(const float* __restrict__ g, const float* __restrict__ q_proj, const T* __restrict__ in_proj_weight,
                   int D, int H, float scale, T* __restrict__ d_in_proj_weight, float* __restrict__ d_q_proj) {
    pdl_wait();
    const int i = blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (i >= D) return;
    const int h = i / (D / H);
    const float* r = g + (static_cast<size_t>(D) + h) * D;
    const float* gv = g + static_cast<size_t>(i) * D;
    const T* wk = in_proj_weight + (static_cast<size_t>(D) + i) * D;
    const float sq = scale * __ldg(q_proj + i);
    T* dwk = d_in_proj_weight ? d_in_proj_weight + (static_cast<size_t>(D) + i) * D : nullptr;
    T* dwv = d_in_proj_weight ? d_in_proj_weight + (2 * static_cast<size_t>(D) + i) * D : nullptr;
    float dot = 0.f;
    for (int d = lane; d < D; d += 32) {
        const float rv = __ldg(r + d);
        dot = fmaf(to_float<T>(wk[d]), rv, dot);
        if (dwk) {
            dwk[d] = from_float<T>(sq * rv);
            dwv[d] = from_float<T>(__ldg(gv + d));
        }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) dot += __shfl_xor_sync(FULL_MASK, dot, off);
    if (lane == 0 && d_q_proj) d_q_proj[i] = scale * dot;
}

// The query-side tail of the backward for a shared query, one launch instead of three (outer product, GEMV, pack):
//   dWq[i, :]  = d_qp[i] * q0[:]                 rows [0, D) of d_in_proj_weight        (torch/nn/functional.py:5854)
//   d_query[i] = sum_k d_qp[k] * Wq[k, i]
//   d_in_proj_bias = [ d_qp | d_bias_kv ]
// Block b owns the 8 indices i = 8b .. 8b+7.  T: the parameters it reads; G: the gradients it writes (the parameter dtype,
// or fp32 next to bf16 shadows of fp32 parameters in mixed precision).
template <typename T, typename G>
__global__ void __launch_bounds__(256)
query_tail_kernel(const float* __restrict__ d_qp, const T* __restrict__ q0, const T* __restrict__ in_proj_weight,
                  const float* __restrict__ d_bias_kv, int D, G* __restrict__ d_in_proj_weight, G* __restrict__ d_query,
                  G* __restrict__ d_in_proj_bias) {
    __shared__ float red[32][9];
    pdl_wait();
    const int i0 = blockIdx.x * 8;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (d_in_proj_weight != nullptr && i0 + warp < D) {
        const int i = i0 + warp;
        const float g = __ldg(d_qp + i);
        G* row = d_in_proj_weight + static_cast<size_t>(i) * D;
        for (int d = lane; d < D; d += 32) row[d] = from_float<G>(g * to_float<T>(q0[d]));
    }
    if (d_query != nullptr) {
        const int ii = threadIdx.x & 7, kl = threadIdx.x >> 3;           // 8 columns x 32 row lanes
        float acc = 0.f;
        if (i0 + ii < D)
            for (int k = kl; k < D; k += 32) acc = fmaf(__ldg(d_qp + k), to_float<T>(in_proj_weight[static_cast<size_t>(k) * D + i0 + ii]), acc);
        red[kl][ii] = acc;
        __syncthreads();
        if (threadIdx.x < 8 && i0 + threadIdx.x < D) {
            float s = 0.f;
#pragma unroll
            for (int k = 0; k < 32; ++k) s += red[k][threadIdx.x];
            d_query[i0 + threadIdx.x] = from_float<G>(s);
        }
    }
    if (d_in_proj_bias != nullptr && threadIdx.x < 8 && i0 + threadIdx.x < D) {
        const int i = i0 + threadIdx.x;
        d_in_proj_bias[i] = from_float<G>(d_qp[i]);
        d_in_proj_bias[D + i] = from_float<G>(d_bias_kv[i]);
        d_in_proj_bias[2 * D + i] = from_float<G>(d_bias_kv[D + i]);
    }
}

int launch_query_tail(int dtype, int grad_dtype, int D, const float* d_qp, const void* q0, const void* in_proj_weight,
                      const float* d_bias_kv, void* d_in_proj_weight, void* d_query, void* d_in_proj_bias, cudaStream_t s) {
    const dim3 grid((D + 7) / 8), block(256);
    if (dtype != grad_dtype) {
        if (dtype != AECF_BF16 || grad_dtype != AECF_F32) return AECF_ERR_INVALID;
        AECF_CUDA_OK(launch_pdl(query_tail_kernel<__nv_bfloat16, float>, grid, block, 0, s, d_qp, static_cast<const __nv_bfloat16*>(q0),
                                static_cast<const __nv_bfloat16*>(in_proj_weight), d_bias_kv, D,
                                static_cast<float*>(d_in_proj_weight), static_cast<float*>(d_query),
                                static_cast<float*>(d_in_proj_bias)));
    } else if (dtype == AECF_BF16)
        AECF_CUDA_OK(launch_pdl(query_tail_kernel<__nv_bfloat16, __nv_bfloat16>, grid, block, 0, s, d_qp, static_cast<const __nv_bfloat16*>(q0),
                                static_cast<const __nv_bfloat16*>(in_proj_weight), d_bias_kv, D,
                                static_cast<__nv_bfloat16*>(d_in_proj_weight), static_cast<__nv_bfloat16*>(d_query),
                                static_cast<__nv_bfloat16*>(d_in_proj_bias)));
    else
        AECF_CUDA_OK(launch_pdl(query_tail_kernel<float, float>, grid, block, 0, s, d_qp, static_cast<const float*>(q0),
                                static_cast<const float*>(in_proj_weight), d_bias_kv, D, static_cast<float*>(d_in_proj_weight),
                                static_cast<float*>(d_query), static_cast<float*>(d_in_proj_bias)));
    count_launch();
    return AECF_OK;
}

static int fold_check(int dtype, int D, int H) {
    if (dtype != AECF_F32 && dtype != AECF_BF16) return AECF_ERR_INVALID;
    if (D <= 0 || H <= 0 || D % H != 0) return AECF_ERR_INVALID;
    if ((static_cast<long long>(D) * D * (dtype == AECF_BF16 ? 2 : 4)) % 16 != 0) return AECF_ERR_UNSUPPORTED;
    return AECF_OK;
}

}  // namespace aecf

using namespace aecf;

extern "C" {

int aecf_fold_prepare(int32_t device, int32_t dtype, int32_t embed_dim, int32_t num_heads, const float* q_proj,
                      const void* in_proj_weight, void* folded_w, void* stream) {
    int rc = fold_check(dtype, embed_dim, num_heads);
    if (rc != AECF_OK) return rc;
    if (!q_proj || !in_proj_weight || !folded_w) return AECF_ERR_INVALID;
    if (!aligned16(in_proj_weight) || !aligned16(folded_w)) return AECF_ERR_ALIGNMENT;
    DeviceScope device_scope__(device);
    if ((rc = device_scope__.rc) != AECF_OK) return rc;
    const int D = embed_dim, H = num_heads, hsp = aecf_fold_score_cols(dtype, H);
    const float scale = static_cast<float>(sqrt(1.0 / static_cast<double>(D / H)));
    const int fold_blocks = hsp * ((D + 31) / 32);
    const int copy_blocks = 128;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    TimedLaunch timed(s);
    if (dtype == AECF_BF16)
        AECF_CUDA_OK(launch_pdl(fold_prepare_kernel<__nv_bfloat16>, dim3(fold_blocks + copy_blocks), dim3(256), 0, s, q_proj,
                                static_cast<const __nv_bfloat16*>(in_proj_weight), D, H, hsp, scale, fold_blocks,
                                static_cast<__nv_bfloat16*>(folded_w)));
    else
        AECF_CUDA_OK(launch_pdl(fold_prepare_kernel<float>, dim3(fold_blocks + copy_blocks), dim3(256), 0, s, q_proj,
                                static_cast<const float*>(in_proj_weight), D, H, hsp, scale, fold_blocks,
                                static_cast<float*>(folded_w)));
    count_launch();
    return AECF_OK;
}

int aecf_fold_prepare_query(int32_t device, int32_t dtype, int32_t embed_dim, int32_t num_heads, const void* query,
                            const void* in_proj_weight, const void* in_proj_bias, float* q_proj, void* folded_w, void* stream) {
    int rc = fold_check(dtype, embed_dim, num_heads);
    if (rc != AECF_OK) return rc;
    if (!query || !in_proj_weight || !q_proj || !folded_w) return AECF_ERR_INVALID;
    if (!aligned16(in_proj_weight) || !aligned16(folded_w) || !aligned16(query)) return AECF_ERR_ALIGNMENT;
    DeviceScope device_scope__(device);
    if ((rc = device_scope__.rc) != AECF_OK) return rc;
    const int D = embed_dim, H = num_heads, hsp = aecf_fold_score_cols(dtype, H);
    const float scale = static_cast<float>(sqrt(1.0 / static_cast<double>(D / H)));
    const int fold_blocks = hsp * ((D + 31) / 32);
    const int copy_blocks = 128;
    const size_t smem = static_cast<size_t>(D / H) * sizeof(float);
    if (smem > 48 * 1024) return AECF_ERR_UNSUPPORTED;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    TimedLaunch timed(s);
    if (dtype == AECF_BF16)
        AECF_CUDA_OK(launch_pdl(fold_prepare_query_kernel<__nv_bfloat16>, dim3(fold_blocks + copy_blocks), dim3(256), smem, s,
                                static_cast<const __nv_bfloat16*>(query), static_cast<const __nv_bfloat16*>(in_proj_weight),
                                static_cast<const __nv_bfloat16*>(in_proj_bias), D, H, hsp, scale, fold_blocks, q_proj,
                                static_cast<__nv_bfloat16*>(folded_w)));
    else
        AECF_CUDA_OK(launch_pdl(fold_prepare_query_kernel<float>, dim3(fold_blocks + copy_blocks), dim3(256), smem, s,
                                static_cast<const float*>(query), static_cast<const float*>(in_proj_weight),
                                static_cast<const float*>(in_proj_bias), D, H, hsp, scale, fold_blocks, q_proj,
                                static_cast<float*>(folded_w)));
    count_launch();
    return AECF_OK;
}

int aecf_fold_finish(int32_t device, int32_t dtype, int32_t embed_dim, int32_t num_heads, const float* g,
                     const float* q_proj, const void* in_proj_weight, void* d_in_proj_weight, float* d_q_proj,
                     void* stream) {
    int rc = fold_check(dtype, embed_dim, num_heads);
    if (rc != AECF_OK) return rc;
    if (!g || !q_proj || !in_proj_weight) return AECF_ERR_INVALID;
    DeviceScope device_scope__(device);
    if ((rc = device_scope__.rc) != AECF_OK) return rc;
    const int D = embed_dim, H = num_heads;
    const float scale = static_cast<float>(sqrt(1.0 / static_cast<double>(D / H)));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    TimedLaunch timed(s);
    if (dtype == AECF_BF16)
        AECF_CUDA_OK(launch_pdl(fold_finish_kernel<__nv_bfloat16>, dim3((D + 7) / 8), dim3(256), 0, s, g, q_proj,
                                static_cast<const __nv_bfloat16*>(in_proj_weight), D, H, scale,
                                static_cast<__nv_bfloat16*>(d_in_proj_weight), d_q_proj));
    else
        AECF_CUDA_OK(launch_pdl(fold_finish_kernel<float>, dim3((D + 7) / 8), dim3(256), 0, s, g, q_proj,
                                static_cast<const float*>(in_proj_weight), D, H, scale, static_cast<float*>(d_in_proj_weight),
                                d_q_proj));
    count_launch();
    return AECF_OK;
}

}  // extern "C"
