// The tail of the folded backward: everything between the tensor-core products and the parameter gradients, in two
// kernels (three with data parallelism) that run on a side stream NEXT TO the dX product instead of eight small launches
// in front of and behind it (r1: colsum x2, split-K reduce x2, pool_bwd_finalize, fold_finish, query_tail = 86 us of a
// 604 us step, all on the critical path).
//
//   grad_gather   raw fp32 sums S = [ [dWv ; R] | dWo | colsum(d_out) | pool bias sums ]: folds the split-K partials of
//                 the two weight-gradient products and leaves per-block column sums of d_out (the gradient of
//                 out_proj.bias, torch/nn/functional.py:6653 backward); grad_fold then folds those and the per-CTA
//                 partials of the pool backward, one warp per column (every load in flight at once: these folds are
//                 latency, not bandwidth)
//   grad_peer_sum (world > 1) S summed over the ranks in fp32 through NVLink peer mappings: flag barrier, rank r sums
//                 slice r of every rank's S in rank order and stores it into every rank's reduced buffer, flag barrier
//                 (the scheme of peer_allreduce.cu, from one buffer into another)
//   grad_finish   S -> parameter gradients in the parameter dtype (fp32 in mixed precision, next to bf16 shadows of the
//                 parameters): dWv, dWk = scale q (x) R, d_qp = scale Wk . R, dWq = d_qp (x) q0, the three in-projection
//                 bias thirds, dWo, d_out_proj_bias; grad_dquery then forms
//                 d_query = d_qp . Wq (reference: what autograd derives from torch/nn/functional.py:5854-5855, 6653 for a
//                 shared query)
//
// Everything downstream of S is linear in S, so summing S over the ranks BEFORE grad_finish gives every rank the gradients
// of the global batch with one rounding to the parameter dtype -- an N-rank run rounds like a 1-rank run (r1 reduced
// bf16-rounded gradients).  S is half the size of the parameter set (dWk, dWq, d_query are images of the H rows of R).
// All reductions are in fixed index order (no atomics).  None of the kernels uses shared memory: they run NEXT TO the dX
// product, whose persistent CTAs leave less than 2 KB of an SM's shared memory (cta_group::2 kernel: 225 KB + the per-CTA
// reserve), and a CTA that needs more would wait for the product to end instead of sharing the SM with it.
#include "common.cuh"
#include "grad_tail.cuh"

namespace aecf {

constexpr int TAIL_THREADS = 256;
template <int N> struct IntTag { static constexpr int value = N; };

// ptxas sinks independent loads next to their uses to save registers (r2 run 6: a batch of 32 loads compiled to four in
// flight); these kernels want the opposite -- every load of a batch issued before the first use -- so the loads are
// volatile and a compiler-level memory barrier separates the issue loop from the consume loop.
#ifdef AECF_CUDA_EMU
__device__ __forceinline__ uint4 ldg_batch(const void* p) { return *reinterpret_cast<const uint4*>(p); }
__device__ __forceinline__ void issue_barrier() {}
#else
__device__ __forceinline__ uint4 ldg_batch(const void* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ void issue_barrier() { asm volatile("" ::: "memory"); }
#endif

// ---- grad_gather / grad_fold ------------------------------------------------------------------------------------------
struct GatherParams {
    const float* g_part; int g_splits; long long g_stride;      // [dWv ; R] partials: g_splits slabs of (D + HSP) * D
    const float* o_part; int o_splits; long long o_stride;      // dWo partials: o_splits slabs of D * D
    const void* d_out; long long rows, ld;                      // [rows, D] in the parameter dtype: column sums -> bo
    // the in-projection bias sums the pool backward no longer forms (pool_bwd.cuh): per sample and head it leaves
    // [s = sum_m wd | sum_m ds] in rowsum [samples][2 HSP]; d_bias_v[d] = sum_b s[b, h(d)] d_ctx[b, d] and
    // d_bias_k[d] = scale q[d] sum_b sum_m ds[b, m, h(d)] (analytically zero; kept as the arithmetic leaves it)
    const float* rowsum; const void* d_ctx; long long samples;
    const float* q_proj; float scale; int head_dim;
    float* pool_part;                                           // [gridDim.x][3 D] scratch: per-block [ - | d_bias_v | d_bias_k ]
    float* sums; TailLayout lay;
    float* colsum_part;                                         // [gridDim.x][D] scratch
    int D, HSP;
};

#ifdef AECF_CUDA_EMU
__device__ __forceinline__ float ldg_batch_f32(const float* p) { return *p; }
#else
__device__ __forceinline__ float ldg_batch_f32(const float* p) {
    float r;
    asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(r) : "l"(p));
    return r;
}
#endif

template <typename T>
__global__ void __launch_bounds__(TAIL_THREADS, 1)
grad_gather_kernel(const GatherParams p) {
    constexpr int V = Vec<T>::N;
    const int t = threadIdx.x;
    const int D = p.D;
    const int NC = D / V;                                       // 16-byte chunks per row of d_out
    pdl_wait();

    // (1) column sums of this block's rows of d_out.  `rl` row lanes (a power of two, lanes of ONE warp, folded by xor
    // shuffles in a fixed order) times 256 / rl chunk columns per pass.
    if (p.d_out != nullptr) {
        int rl = 32;
        while (rl > 1 && TAIL_THREADS / rl < NC) rl >>= 1;      // as many row lanes as still cover a row in one pass, if possible
        const int ncp = TAIL_THREADS / rl;                      // chunk columns per pass
        const int lane_r = t % rl, cc = t / rl;
        const long long per = (p.rows + gridDim.x - 1) / gridDim.x;
        const long long r0 = per * blockIdx.x, r1 = min(p.rows, r0 + per);
        const T* x = static_cast<const T*>(p.d_out);
        for (int cb = 0; cb < NC; cb += ncp) {
            const bool active = cb + cc < NC;
            float acc[V];
#pragma unroll
            for (int v = 0; v < V; ++v) acc[v] = 0.f;
            if (active) {
                const T* col = x + static_cast<long long>(cb + cc) * V;
                // 16 rows in flight per thread: next to a tensor-core product a trip to memory takes several microseconds,
                // and what this kernel costs is the number of trips (r2 run 6: 26 us alone, 4x that next to a product at U = 8)
                long long r = r0 + lane_r;
                auto batch = [&](auto tag) {                    // tag.value rows in flight at once
                    constexpr int U = decltype(tag)::value;
                    for (; r + static_cast<long long>(U - 1) * rl < r1; r += static_cast<long long>(U) * rl) {
                        uint4 raw[U];
#pragma unroll
                        for (int u = 0; u < U; ++u) raw[u] = ldg_batch(col + (r + static_cast<long long>(u) * rl) * p.ld);
                        issue_barrier();
#pragma unroll
                        for (int u = 0; u < U; ++u) {
                            float f[V];
                            Vec<T>::unpack(raw[u], f);
#pragma unroll
                            for (int v = 0; v < V; ++v) acc[v] += f[v];
                        }
                    }
                };
                batch(IntTag<16>{});
                batch(IntTag<4>{});
                batch(IntTag<1>{});
            }
            for (int off = rl >> 1; off > 0; off >>= 1) {       // the rl row lanes are neighbouring lanes of one warp
#pragma unroll
                for (int v = 0; v < V; ++v) acc[v] += __shfl_xor_sync(FULL_MASK, acc[v], off);
            }
            if (active && lane_r == 0) {
                float* out = p.colsum_part + static_cast<long long>(blockIdx.x) * D + static_cast<long long>(cb + cc) * V;
#pragma unroll
                for (int v = 0; v < V; ++v) out[v] = acc[v];
            }
        }
    }

    // (1b) the same walk over d_ctx, every row weighted per head: this block's share of d_bias_v and d_bias_k
    if (p.rowsum != nullptr) {
        int rl = 32;
        while (rl > 1 && TAIL_THREADS / rl < NC) rl >>= 1;
        const int ncp = TAIL_THREADS / rl;
        const int lane_r = t % rl, cc = t / rl;
        const long long per = (p.samples + gridDim.x - 1) / gridDim.x;
        const long long r0 = per * blockIdx.x, r1 = min(p.samples, r0 + per);
        const T* x = static_cast<const T*>(p.d_ctx);
        const long long wld = 2LL * p.HSP;
        for (int cb = 0; cb < NC; cb += ncp) {
            const bool active = cb + cc < NC;
            float acc[V], acc_k = 0.f;
#pragma unroll
            for (int v = 0; v < V; ++v) acc[v] = 0.f;
            if (active) {
                const T* col = x + static_cast<long long>(cb + cc) * V;
                const float* wcol = p.rowsum + ((cb + cc) * V) / p.head_dim;     // this chunk's head
                long long r = r0 + lane_r;
                auto batch = [&](auto tag) {
                    constexpr int U = decltype(tag)::value;
                    for (; r + static_cast<long long>(U - 1) * rl < r1; r += static_cast<long long>(U) * rl) {
                        uint4 raw[U];
                        float ws[U], wk[U];
#pragma unroll
                        for (int u = 0; u < U; ++u) {
                            const long long rr = r + static_cast<long long>(u) * rl;
                            raw[u] = ldg_batch(col + rr * D);
                            ws[u] = ldg_batch_f32(wcol + rr * wld);
                            wk[u] = ldg_batch_f32(wcol + rr * wld + p.HSP);
                        }
                        issue_barrier();
#pragma unroll
                        for (int u = 0; u < U; ++u) {
                            float f[V];
                            Vec<T>::unpack(raw[u], f);
#pragma unroll
                            for (int v = 0; v < V; ++v) acc[v] = fmaf(ws[u], f[v], acc[v]);
                            acc_k += wk[u];
                        }
                    }
                };
                batch(IntTag<8>{});
                batch(IntTag<1>{});
            }
            for (int off = rl >> 1; off > 0; off >>= 1) {
#pragma unroll
                for (int v = 0; v < V; ++v) acc[v] += __shfl_xor_sync(FULL_MASK, acc[v], off);
                acc_k += __shfl_xor_sync(FULL_MASK, acc_k, off);
            }
            if (active && lane_r == 0) {
                const int c = (cb + cc) * V;
                float* out = p.pool_part + static_cast<long long>(blockIdx.x) * 3 * D;
#pragma unroll
                for (int v = 0; v < V; ++v) {
                    out[D + c + v] = acc[v];
                    out[2 * D + c + v] = p.scale * __ldg(p.q_proj + c + v) * acc_k;
                }
            }
        }
    }

    // (2) split-K partials of the two weight-gradient products, splits in order, 16 bytes per thread, four splits in flight
    const long long gt = static_cast<long long>(blockIdx.x) * TAIL_THREADS + t;
    const long long nthreads = static_cast<long long>(gridDim.x) * TAIL_THREADS;
    auto fold = [&](const float* part, int splits, long long stride, long long n, float* out) {
        if (part == nullptr) return;
        for (long long i = gt; i < n / 4; i += nthreads) {
            float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
            int z = 0;
            for (; z + 8 <= splits; z += 8) {
                uint4 v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) v[u] = ldg_batch(part + (z + u) * stride + 4 * i);
                issue_barrier();
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    s.x += __uint_as_float(v[u].x); s.y += __uint_as_float(v[u].y);
                    s.z += __uint_as_float(v[u].z); s.w += __uint_as_float(v[u].w);
                }
            }
            if (z < splits) {                                   // the rest, also in one trip
                uint4 v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) v[u] = (z + u < splits) ? ldg_batch(part + (z + u) * stride + 4 * i) : make_uint4(0, 0, 0, 0);
                issue_barrier();
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    s.x += __uint_as_float(v[u].x); s.y += __uint_as_float(v[u].y);
                    s.z += __uint_as_float(v[u].z); s.w += __uint_as_float(v[u].w);
                }
                z = splits;
            }
            for (; z < splits; ++z) {
                const float4 v = *reinterpret_cast<const float4*>(part + z * stride + 4 * i);
                s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
            }
            *reinterpret_cast<float4*>(out + 4 * i) = s;
        }
    };
    fold(p.g_part, p.g_splits, p.g_stride, static_cast<long long>(D + p.HSP) * D, p.sums + p.lay.g);
    fold(p.o_part, p.o_splits, p.o_stride, static_cast<long long>(D) * D, p.sums + p.lay.o);
}

// One warp per column: lane l sums rows l, l + 32, ... (every load issued before the first add), the 32 lane sums are
// folded by xor shuffles.  Columns [0, D): the per-block column sums of d_out -> bo; columns [D, 4 D): the pool backward's
// per-block in-projection bias sums [ - | d_bias_v | d_bias_k] of grad_gather -> pool.
struct FoldParams {
    const float* colsum_part; int colsum_rows;                  // [colsum_rows][D], or null
    const float* pool_part; int pool_rows;                      // [pool_rows][3 D], or null; the first third is not written (folded)
    float* sums; TailLayout lay;
    int D;
};

__global__ void __launch_bounds__(512, 1)
grad_fold_kernel(const FoldParams p) {
    const int lane = threadIdx.x & 31;
    const int col = blockIdx.x * 16 + (threadIdx.x >> 5);
    pdl_wait();
    if (col >= 4 * p.D) return;
    if (col >= p.D && col < 2 * p.D) {                          // (the d_q third of the unfolded layout: unused here)
        if (lane == 0) p.sums[p.lay.pool + col - p.D] = 0.f;
        return;
    }
    const bool is_colsum = col < p.D;
    const float* part = is_colsum ? p.colsum_part : p.pool_part;
    if (part == nullptr) return;
    const int rows = is_colsum ? p.colsum_rows : p.pool_rows;
    const long long ld = is_colsum ? p.D : 3LL * p.D;
    const int c = is_colsum ? col : col - p.D;
    float s = 0.f;
    constexpr int U = 16;
    for (int r0 = lane; r0 < rows; r0 += 32 * U) {
        float v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int r = r0 + 32 * u;
            v[u] = r < rows ? part[static_cast<long long>(r) * ld + c] : 0.f;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) s += v[u];
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(FULL_MASK, s, off);
    if (lane == 0) p.sums[(is_colsum ? p.lay.bo : p.lay.pool) + c] = s;
}

// ---- grad_finish / grad_dquery ----------------------------------------------------------------------------------------
struct FinishParams {
    const float* sums; TailLayout lay;
    const float* q_proj;            // [D] fp32: projected query (unscaled)
    const void* in_proj_weight;     // [3D, D]
    const void* query;              // [D]
    const void* out_proj_weight;    // [D, D] or null; non-null: d_bias_v = Wo^T colsum(d_out), d_bias_k = 0 (pool_bwd.cuh)
    void* d_in_w;                   // [3D, D], nullable
    void* d_in_b;                   // [3D], nullable
    void* d_out_w;                  // [D, D], nullable
    void* d_out_b;                  // [D], nullable
    void* d_query;                  // [D], nullable
    float* d_qp;                    // [ceil(D / 8)][D] scratch: per-block partials of d_query
    int D, H, HSP;
    float scale;
};

template <typename T> __device__ __forceinline__ void store4(T* p, float a, float b, float c, float d);
template <> __device__ __forceinline__ void store4<float>(float* p, float a, float b, float c, float d) {
    *reinterpret_cast<float4*>(p) = make_float4(a, b, c, d);
}
template <> __device__ __forceinline__ void store4<__nv_bfloat16>(__nv_bfloat16* p, float a, float b, float c, float d) {
    *reinterpret_cast<uint2*>(p) = make_uint2(Vec<__nv_bfloat16>::pack2(a, b), Vec<__nv_bfloat16>::pack2(c, d));
}
template <typename T> __device__ __forceinline__ float4 load4(const T* p);
template <> __device__ __forceinline__ float4 load4<float>(const float* p) { return *reinterpret_cast<const float4*>(p); }
template <> __device__ __forceinline__ float4 load4<__nv_bfloat16>(const __nv_bfloat16* p) {
    const uint2 r = *reinterpret_cast<const uint2*>(p);
    return make_float4(__uint_as_float(r.x << 16), __uint_as_float(r.x & 0xffff0000u), __uint_as_float(r.y << 16),
                       __uint_as_float(r.y & 0xffff0000u));
}

// One warp per in-projection row i (head h = i / head_dim), 8 rows per block:
//   dWv[i, :] = G[i, :]     dWk[i, :] = scale q[i] R[h, :]     d_qp[i] = scale Wk[i, :] . R[h, :]     dWo[i, :] = O[i, :]
//   dWq[i, :] = d_qp[i] q0[:]     d_in_b = [ d_qp | d_bias_k | d_bias_v ]     d_out_b = colsum(d_out)
// T: the parameters it reads (in_proj_weight, query, out_proj_weight); TG: the parameter gradients it writes (fp32 in mixed
// precision, where the parameters are bf16 shadows of fp32 masters).
template <typename T, typename TG>
__global__ void __launch_bounds__(TAIL_THREADS, 1)
grad_finish_kernel(const FinishParams p) {
    __shared__ float qps[8];                                    // d_qp of the block's 8 rows
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int D = p.D;
    const int i = blockIdx.x * 8 + warp;
    pdl_wait();
    const T* W = static_cast<const T*>(p.in_proj_weight);
    const T* q0 = static_cast<const T*>(p.query);
    TG* d_in_w = static_cast<TG*>(p.d_in_w);
    float d_qp = 0.f;
    if (i < D) {
    const int h = i / (D / p.H);
    const float* R = p.sums + p.lay.g + static_cast<long long>(D + h) * D;
    const float* G = p.sums + p.lay.g + static_cast<long long>(i) * D;
    const float* O = p.sums + p.lay.o + static_cast<long long>(i) * D;
    const T* wk = W + (static_cast<long long>(D) + i) * D;
    const float sq = p.scale * __ldg(p.q_proj + i);
    float dot = 0.f;
    // four 128-column steps (one 512-wide batch) at a time: every load of the batch is issued before anything is stored, so a
    // row costs one trip to memory, not four (the kernel is nothing but latency)
    for (int d0 = lane * 4; d0 < D; d0 += 512) {
        float4 r[4], w[4], g[4], o[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int d = d0 + 128 * u;
            const bool ok = d < D;
            r[u] = ok ? *reinterpret_cast<const float4*>(R + d) : make_float4(0.f, 0.f, 0.f, 0.f);
            w[u] = ok ? load4<T>(wk + d) : make_float4(0.f, 0.f, 0.f, 0.f);
            g[u] = (ok && d_in_w != nullptr) ? *reinterpret_cast<const float4*>(G + d) : make_float4(0.f, 0.f, 0.f, 0.f);
            o[u] = (ok && p.d_out_w != nullptr) ? *reinterpret_cast<const float4*>(O + d) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int d = d0 + 128 * u;
            if (d >= D) continue;
            dot = fmaf(w[u].x, r[u].x, dot); dot = fmaf(w[u].y, r[u].y, dot);
            dot = fmaf(w[u].z, r[u].z, dot); dot = fmaf(w[u].w, r[u].w, dot);
            if (d_in_w != nullptr) {
                store4<TG>(d_in_w + (static_cast<long long>(D) + i) * D + d, sq * r[u].x, sq * r[u].y, sq * r[u].z, sq * r[u].w);
                store4<TG>(d_in_w + (2LL * D + i) * D + d, g[u].x, g[u].y, g[u].z, g[u].w);
            }
            if (p.d_out_w != nullptr)
                store4<TG>(static_cast<TG*>(p.d_out_w) + static_cast<long long>(i) * D + d, o[u].x, o[u].y, o[u].z, o[u].w);
        }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) dot += __shfl_xor_sync(FULL_MASK, dot, off);
    d_qp = p.scale * dot;
    if (d_in_w != nullptr) {
        for (int d0 = lane * 4; d0 < D; d0 += 512) {
            float4 q[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) q[u] = (d0 + 128 * u < D) ? load4<T>(q0 + d0 + 128 * u) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (d0 + 128 * u < D)
                    store4<TG>(d_in_w + static_cast<long long>(i) * D + d0 + 128 * u, d_qp * q[u].x, d_qp * q[u].y, d_qp * q[u].z,
                              d_qp * q[u].w);
        }
    }
    float bias_v = 0.f;
    if (p.d_in_b != nullptr && p.out_proj_weight != nullptr) {  // column i of Wo against the column sums of d_out
        const T* wo = static_cast<const T*>(p.out_proj_weight) + i;
        const float* bo = p.sums + p.lay.bo;
        constexpr int U = 16;
        for (int j0 = lane; j0 < D; j0 += 32 * U) {
            float w[U], b[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int j = j0 + 32 * u;
                w[u] = j < D ? to_float<T>(wo[static_cast<long long>(j) * D]) : 0.f;
                b[u] = j < D ? bo[j] : 0.f;
            }
#pragma unroll
            for (int u = 0; u < U; ++u) bias_v = fmaf(w[u], b[u], bias_v);
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) bias_v += __shfl_xor_sync(FULL_MASK, bias_v, off);
    }
    if (lane == 0) {
        if (p.d_in_b != nullptr) {
            TG* db = static_cast<TG*>(p.d_in_b);
            db[i] = from_float<TG>(d_qp);
            if (p.out_proj_weight != nullptr) {
                db[D + i] = from_float<TG>(0.f);                                    // d_bias_k
                db[2 * D + i] = from_float<TG>(bias_v);                             // d_bias_v
            } else {
                db[D + i] = from_float<TG>(p.sums[p.lay.pool + 2LL * D + i]);       // d_bias_k
                db[2 * D + i] = from_float<TG>(p.sums[p.lay.pool + D + i]);         // d_bias_v
            }
        }
        if (p.d_out_b != nullptr) static_cast<TG*>(p.d_out_b)[i] = from_float<TG>(p.sums[p.lay.bo + i]);
    }
    }   // i < D
    // this block's share of d_query[c] = sum_i d_qp[i] Wq[i, c] (torch/nn/functional.py:5854 backward): a thread owns its
    // columns and sums the block's 8 rows in order, all 8 loads in flight; grad_dquery_fold sums the blocks
    if (p.d_query == nullptr) return;
    if (lane == 0) qps[warp] = d_qp;                            // rows past D contribute 0
    __syncthreads();
    const int rows = min(8, D - static_cast<int>(blockIdx.x) * 8);
    for (int c = threadIdx.x; c < D; c += TAIL_THREADS) {
        float w[8];
#pragma unroll
        for (int k = 0; k < 8; ++k)
            w[k] = k < rows ? to_float<T>(W[(static_cast<long long>(blockIdx.x) * 8 + k) * D + c]) : 0.f;
        float s = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) s = fmaf(qps[k], w[k], s);
        p.d_qp[static_cast<long long>(blockIdx.x) * D + c] = s;
    }
}

// d_query[c] = sum over the blocks of grad_finish of their partials: one warp per column, every load in flight at once.
template <typename T>
__global__ void __launch_bounds__(TAIL_THREADS, 1)
grad_dquery_fold_kernel(const float* __restrict__ part, int rows, int D, T* __restrict__ d_query) {
    const int lane = threadIdx.x & 31;
    const int c = blockIdx.x * (TAIL_THREADS / 32) + (threadIdx.x >> 5);
    pdl_wait();
    if (c >= D) return;
    float s = 0.f;
    constexpr int U = 8;
    for (int r0 = lane; r0 < rows; r0 += 32 * U) {
        float v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) v[u] = (r0 + 32 * u < rows) ? part[static_cast<long long>(r0 + 32 * u) * D + c] : 0.f;
#pragma unroll
        for (int u = 0; u < U; ++u) s += v[u];
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(FULL_MASK, s, off);
    if (lane == 0) d_query[c] = from_float<T>(s);
}

// ---- host side ----------------------------------------------------------------------------------------------------------
static size_t align256(size_t x) { return (x + 255) & ~static_cast<size_t>(255); }

size_t grad_tail_scratch_bytes(int D, int sms) {
    return align256(static_cast<size_t>(sms) * D * sizeof(float))           // per-block column sums of d_out
         + align256(static_cast<size_t>((D + 7) / 8) * D * sizeof(float))   // per-block partials of d_query
         + align256(static_cast<size_t>(sms) * 3 * D * sizeof(float));      // per-block in-projection bias sums
}

// which = GATHER_EARLY: column sums of d_out (per block) and the dWo fold -- everything the backward knows after its first
// product; GATHER_LATE: the [dWv ; R] fold, then grad_fold (the column-sum and pool partials -> S).
int launch_grad_gather(const GradTailArgs& a, int which, cudaStream_t s) {
    const int V = a.dtype == AECF_BF16 ? 8 : 4;
    if (a.D % V != 0) return AECF_ERR_UNSUPPORTED;
    const TailLayout lay = tail_layout(a.D, a.HSP);
    // at most one block per SM: two of them take the 2 KB of shared memory a product's CTA leaves, and a persistent CTA
    // that cannot start on its SM delays the whole product by as long as it waits (r2 run 6: dX 116 -> 134 us)
    const int blocks = a.sms;
    GatherParams p{};
    p.sums = a.sums; p.lay = lay; p.D = a.D; p.HSP = a.HSP;
    p.colsum_part = static_cast<float*>(a.scratch);
    const bool early = which == GATHER_EARLY;
    float* pool_part = reinterpret_cast<float*>(static_cast<char*>(a.scratch) + align256(static_cast<size_t>(a.sms) * a.D * sizeof(float))
                                                + align256(static_cast<size_t>((a.D + 7) / 8) * a.D * sizeof(float)));
    if (early) {
        p.o_part = a.o.partial; p.o_splits = a.o.splits; p.o_stride = a.o.stride;
        p.d_out = a.d_out; p.rows = a.rows; p.ld = a.D;
        if (a.rowsum != nullptr && a.d_ctx != nullptr) {
            p.rowsum = a.rowsum; p.d_ctx = a.d_ctx; p.samples = a.samples; p.q_proj = a.q_proj;
            p.head_dim = a.D / a.H;
            p.scale = static_cast<float>(sqrt(1.0 / static_cast<double>(a.D / a.H)));
            p.pool_part = pool_part;
        }
    } else {
        p.g_part = a.g.partial; p.g_splits = a.g.splits; p.g_stride = a.g.stride;
    }
    TimedLaunch timed(s, AECF_SITE_GRAD_GATHER);
    if (p.o_part != nullptr || p.d_out != nullptr || p.g_part != nullptr || p.rowsum != nullptr) {
        if (a.dtype == AECF_BF16) AECF_CUDA_OK(launch_pdl(grad_gather_kernel<__nv_bfloat16>, dim3(blocks), dim3(TAIL_THREADS), 0, s, p));
        else AECF_CUDA_OK(launch_pdl(grad_gather_kernel<float>, dim3(blocks), dim3(TAIL_THREADS), 0, s, p));
        count_launch();
    }
    if (!early) {
        FoldParams f{};
        f.colsum_part = a.d_out ? p.colsum_part : nullptr; f.colsum_rows = blocks;
        f.pool_part = (a.rowsum != nullptr && a.d_ctx != nullptr) ? pool_part : nullptr; f.pool_rows = blocks;
        f.sums = a.sums; f.lay = lay; f.D = a.D;
        AECF_CUDA_OK(launch_pdl(grad_fold_kernel, dim3((4 * a.D + 15) / 16), dim3(512), 0, s, f));
        count_launch();
    }
    return AECF_OK;
}

int launch_grad_finish(const GradTailArgs& a, const float* sums, cudaStream_t s) {
    if (a.D % 4 != 0) return AECF_ERR_UNSUPPORTED;
    if (a.dtype != a.grad_dtype && (a.dtype != AECF_BF16 || a.grad_dtype != AECF_F32)) return AECF_ERR_INVALID;
    FinishParams p{};
    p.sums = sums; p.lay = tail_layout(a.D, a.HSP);
    p.q_proj = a.q_proj; p.in_proj_weight = a.in_proj_weight; p.query = a.query; p.out_proj_weight = a.out_proj_weight;
    p.d_in_w = a.d_in_w; p.d_in_b = a.d_in_b; p.d_out_w = a.d_out_w; p.d_out_b = a.d_out_b; p.d_query = a.d_query;
    p.D = a.D; p.H = a.H; p.HSP = a.HSP;
    p.scale = static_cast<float>(sqrt(1.0 / static_cast<double>(a.D / a.H)));
    p.d_qp = reinterpret_cast<float*>(static_cast<char*>(a.scratch) + align256(static_cast<size_t>(a.sms) * a.D * sizeof(float)));
    const dim3 grid(static_cast<unsigned>((a.D + 7) / 8)), block(TAIL_THREADS);
    TimedLaunch timed(s, AECF_SITE_GRAD_FINISH);
    if (a.dtype != a.grad_dtype) AECF_CUDA_OK(launch_pdl(grad_finish_kernel<__nv_bfloat16, float>, grid, block, 0, s, p));
    else if (a.dtype == AECF_BF16) AECF_CUDA_OK(launch_pdl(grad_finish_kernel<__nv_bfloat16, __nv_bfloat16>, grid, block, 0, s, p));
    else AECF_CUDA_OK(launch_pdl(grad_finish_kernel<float, float>, grid, block, 0, s, p));
    count_launch();
    if (a.d_query != nullptr) {                                 // (reads fp32 partials only: one type, the gradient's)
        const dim3 g2(static_cast<unsigned>((a.D + 7) / 8));
        const int rows = (a.D + 7) / 8;
        if (a.grad_dtype == AECF_BF16)
            AECF_CUDA_OK(launch_pdl(grad_dquery_fold_kernel<__nv_bfloat16>, g2, block, 0, s, static_cast<const float*>(p.d_qp), rows, a.D,
                                    static_cast<__nv_bfloat16*>(a.d_query)));
        else
            AECF_CUDA_OK(launch_pdl(grad_dquery_fold_kernel<float>, g2, block, 0, s, static_cast<const float*>(p.d_qp), rows, a.D,
                                    static_cast<float*>(a.d_query)));
        count_launch();
    }
    return AECF_OK;
}

}  // namespace aecf
