// Shared core of the fused pool kernels.
//
// Work split (DESIGN.md "pool kernels").  A row of D elements is cut into NC = D / V chunks of
// V = 16 bytes / sizeof(T) elements.  A warp owns a SLICE of 32*J consecutive chunks of one
// sample (J = 1, 2 or 4 chunk columns; lane l holds chunks l, l+32, ... of the slice), so every
// warp-wide load instruction covers 512 contiguous bytes.  WPS = ceil(NC / (32 J)) warps share a
// sample; at the headline shape (D = 512, bf16) one warp owns the whole sample.
// A head spans G = head_dim / V consecutive chunks: for G <= 32 it is an aligned group of G lanes
// inside one chunk column, for G > 32 it is all 32 lanes of R = G / 32 consecutive columns
// (R <= J, so a head never straddles warps).  Per-head dot products are segmented xor-shuffle
// reductions; afterwards every lane of a head holds the head's value.
// Heads of GR chunks with GR not a power of two (head_dim 48, 80, 96, ...: the PAD instantiations) are
// padded in the lane map to G = the next power of two: slices, J and WPS are then those of a VIRTUAL row
// of H * G chunks, virtual chunk v belongs to head v >> logG at offset o = v & (G - 1), and it is real chunk
// (v >> logG) * GR + o when o < GR, else an idle lane that loads zeros, joins its head's butterflies
// and stores nothing.  Everything per head (butterflies, head sums, Philox keys) is the same code for
// both maps; only addresses, validity tests and the indices of real columns go through the map.
// Heads are independent everywhere except the head-mean of the forward (and of the eval-mode
// entropy gradient), which crosses warps through shared memory when WPS > 1.
#pragma once

#include <cstddef>

#include "common.cuh"

namespace aecf {

constexpr int POOL_WARPS = 8;               // warps per CTA for both directions

struct PoolParams {
    long long B;
    int D, H, NC, G, logG, LG, R;           // LG = min(G, 32) lanes per head group, R = max(1, G / 32); G = 2^logG is the
                                            // head's span in the lane map (padded map: GR rounded up, see the end)
    int WPS, SPC;                           // warps per sample, samples per CTA (WPS * SPC = POOL_WARPS)
    float scale, p_drop, one_minus_p, base_mask_prob, log_m;   // one_minus_p = float(1.0 - double(p_drop))
    int training, masking, min_active, q_shared;   // masking: 0 off, 1 training-mode stage, 2 eval-mode stage
    RngKey rng;
    const unsigned long long* rng_state;    // device {seed, offset} overriding rng.k0/k1/offset (graph capture), or null
    const void* q;
    const void* kv;
    const float* bias;
    long long bias_sb, bias_sh;
    long long kv_sb, kv_sm;                 // kv element strides between rows / tokens
    long long dkv_sb, dkv_sm;               // d_kv element strides (the same, except in the folded layout)
    // folded key projection (FOLD kernels, DESIGN.md): kv holds the projected VALUES only ([*, D] rows, the V
    // "half" sits at offset 0), the scaled per-head scores come precomputed, and d_kv rows are [dV (D) | ds (HSP)]
    const float* scores;                    // [*, HS] fp32, element (b, m, h) at b*s_sb + m*s_sm + h
    long long s_sb, s_sm;
    int HSP;                                // score-gradient columns per d_kv row (H rounded up to 16 bytes)
    // forward outputs
    void* ctx;
    float* pooled;
    float* entropy;
    float* mask_rate;
    float* masked;
    uint8_t* mask_bits;
    // backward
    const void* d_ctx;
    const float* d_pooled;
    const float* d_entropy;
    void* d_kv;
    void* d_q;
    float* partials;                        // [grid][3][D] fp32: dq | dbv | dbk (folded key projection: the first third is not written)
    float* rowsum;                          // backward, folded: [src_rows][2 HSP] fp32 per-sample sums [s | sum_m ds] (see pool_bwd.cuh), or null
    long long chunk;                        // backward: samples per CTA (CTA b owns [b * chunk, (b + 1) * chunk)); 0: grid-stride
    // Row indirection (aecf_pool_desc::row_index): row i of this call -- its Philox row, its info outputs, d_pooled /
    // d_entropy -- is SAMPLE row_index[i] of the kv / scores / ctx / d_ctx / d_kv buffers (the reference's x-ray model pools
    // only the rows where both modalities are present, xrays/train_xrays_example.py:202-222).  Null: the identity.
    const long long* row_index;
    // fused CurriculumMasking.entropy_loss (streaming forward kernel only; include/aecf_b200.h aecf_pool_desc::loss_out)
    float* loss_out;                        // [1], or null
    float* loss_partials;                   // [gridDim.x] per-CTA sums of (scrubbed entropy - target)^2
    unsigned* loss_ticket;                  // [2]: CTAs done; zero on entry and on exit
    float loss_target;
    // padded lane map (PoolCore<..., PAD = true>): GR real chunks per head (power-of-two heads: GR = G; only the PAD
    // instantiations read it).  It fills the 4 bytes of tail padding behind loss_target: sizeof(PoolParams) is unchanged,
    // and with it the code of the existing kernels (a larger parameter block changes their register allocation).
    int GR;
};
static_assert(sizeof(PoolParams) % 8 == 0 && offsetof(PoolParams, GR) + sizeof(int) == sizeof(PoolParams),
              "GR must sit in the tail padding of PoolParams");

constexpr int POOL_LOSS_MAX_CTAS = 4096;    // loss workspace: POOL_LOSS_MAX_CTAS floats + 64 bytes of counters

__device__ __forceinline__ float scrub_entropy(float e, bool* finite) {     // torch.nan_to_num(nan=0, posinf=1, neginf=0)
    *finite = fabsf(e) <= 3.402823466e38f;
    if (*finite) return e;
    return (e == INFINITY) ? 1.0f : 0.0f;
}

// Several fusion queries per sample (pool_multi.cuh): the S rows (b, 0 .. S-1) share the kv rows of sample b.
// Info outputs, d_pooled, d_entropy and the Philox row are indexed b*S + s.  A second kernel argument, so that
// PoolParams -- and with it the parameter layout of the single-query kernels -- stays as measured.
struct MultiQuery {
    int S;
    long long q_rb, q_rs;                   // row of (b, s) in q / ctx / d_ctx / d_q: b*q_rb + s*q_rs
    const float* bias;                      // additive score bias (PoolParams::bias stays null in this mode) ...
    long long bias_sb, bias_sh, bias_ss;    // ... element (b, h, s, m) at b*bias_sb + h*bias_sh + s*bias_ss + m
};

__device__ __forceinline__ long long source_row(const PoolParams& p, long long row) {
    return p.row_index != nullptr ? __ldg(p.row_index + row) : row;
}

// PAD: the padded lane map (head of GR chunks, GR not a power of two; see the top of the file).  PAD = false is the
// power-of-two map, and every function below reduces to the same expression it has always been for it.
template <typename T, int M, int J, bool DROP, bool PAD = false>
struct PoolCore {
    static constexpr int V = Vec<T>::N;
    static constexpr int CPW = 32 * J;               // chunks per warp slice

    // ---- lane map: the lane with first chunk c0 owns the (virtual) chunks c0 + 32 j, j < J --------------------------
    // real chunk of virtual chunk v (meaningful when v is valid)
    static __device__ __forceinline__ int real_chunk(const PoolParams& p, int v) {
        if constexpr (PAD) return (v >> p.logG) * p.GR + (v & (p.G - 1));
        else return v;
    }
    // virtual chunk of real chunk c (the per-warp strips are laid out by virtual chunk)
    static __device__ __forceinline__ int virtual_chunk(const PoolParams& p, int c) {
        if constexpr (PAD) return ((c / p.GR) << p.logG) + c % p.GR;
        else return c;
    }
    // column j of this lane holds a real chunk ...
    static __device__ __forceinline__ bool valid(const PoolParams& p, int c0, int j) {
        if constexpr (PAD) return c0 + 32 * j < (p.H << p.logG) && ((c0 + 32 * j) & (p.G - 1)) < p.GR;
        else return c0 + 32 * j < p.NC;
    }
    // ... or at least lies inside a head (an idle padding lane still holds its head's reduced values)
    static __device__ __forceinline__ bool in_head(const PoolParams& p, int c0, int j) {
        if constexpr (PAD) return c0 + 32 * j < (p.H << p.logG);
        else return c0 + 32 * j < p.NC;
    }
    // byte offset of this lane's column-0 chunk inside a row, and of its column j relative to that.  Padded: 32 lanes
    // still cover 32 / G whole heads = 32 GR / G contiguous real chunks, so a warp access stays one contiguous run.
    // Column j starts 32 j virtual chunks after column 0 at the same offset inside a head (G <= 32), or at offset + 32 j
    // inside the same slice of heads (G > 32: slices start on head boundaries): either way real_chunk(32 j) real chunks
    // further, the same for every lane, so the offsets stay in uniform registers.
    static __device__ __forceinline__ size_t lane_bytes(const PoolParams& p, int c0) {
        return static_cast<size_t>(real_chunk(p, c0)) * 16;
    }
    static __device__ __forceinline__ int col_bytes(const PoolParams& p, int c0, int j) {
        if constexpr (PAD) return real_chunk(p, 32 * j) * 16;
        else return j * 512;
    }

    // byte offset of this lane's first chunk (c0) of `row` inside kv / d_kv ...
    static __device__ __forceinline__ size_t row_offset(const PoolParams& p, long long row, int c0) {
        return static_cast<size_t>(row) * p.kv_sb * sizeof(T) + lane_bytes(p, c0);
    }
    // ... and, relative to it, of chunk column j of the K half (half = 0) or V half (half = 1) of token m.  64-bit: in a
    // sequence-first layout the token stride is B * 2D elements, so (M - 1) tokens span more than 2^31 bytes at large B.
    static __device__ __forceinline__ long long kv_rel(const PoolParams& p, int c0, int m, int half, int j) {
        return (m * p.kv_sm + half * p.D) * static_cast<long long>(sizeof(T)) + col_bytes(p, c0, j);
    }

    // the same two offsets inside d_kv (its rows are wider than kv's in the folded layout)
    static __device__ __forceinline__ size_t drow_offset(const PoolParams& p, long long row, int c0) {
        return static_cast<size_t>(row) * p.dkv_sb * sizeof(T) + lane_bytes(p, c0);
    }
    static __device__ __forceinline__ long long dkv_rel(const PoolParams& p, int c0, int m, int half, int j) {
        return (m * p.dkv_sm + half * p.D) * static_cast<long long>(sizeof(T)) + col_bytes(p, c0, j);
    }

    // This lane's chunks of `row` of a [rows][D] buffer (ctx, d_ctx).  The power-of-two map keeps the spelling it was
    // measured with: the same arithmetic through col_bytes changes the register allocation of some of its instantiations,
    // J = 1 above all (scripts/sass_diff.py).  The weighted value sums and the ctx stores stay inline in each forward
    // kernel: as shared helpers they changed the SASS of 525 of the 1056 forward kernels (sums) and of slice and
    // streaming kernels (stores).
    static __device__ __forceinline__ void load_row(const PoolParams& p, const void* base, long long row, int c0,
                                                    uint4 (&raw)[J]) {
        const char* in = static_cast<const char*>(base) + static_cast<size_t>(row) * p.D * sizeof(T) + lane_bytes(p, c0);
        if constexpr (PAD) {
#pragma unroll
            for (int j = 0; j < J; ++j) raw[j] = valid(p, c0, j) ? ldg_stream(in + col_bytes(p, c0, j)) : make_uint4(0, 0, 0, 0);
        } else {
#pragma unroll
            for (int j = 0; j < J; ++j) raw[j] = valid(p, c0, j) ? ldg_stream(in + j * 512) : make_uint4(0, 0, 0, 0);
        }
    }

    // projected query chunks, pre-multiplied by scale (torch/nn/functional.py:6632)
    static __device__ __forceinline__ void load_query(const PoolParams& p, long long row, int c0, float (&qs)[J][V]) {
#pragma unroll
        for (int j = 0; j < J; ++j) {
            const int c = real_chunk(p, c0 + 32 * j);
#pragma unroll
            for (int v = 0; v < V; ++v) qs[j][v] = 0.f;
            if (valid(p, c0, j)) {
                if (p.q_shared) {
                    const float* q = static_cast<const float*>(p.q) + static_cast<size_t>(c) * V;
#pragma unroll
                    for (int v4 = 0; v4 < V; v4 += 4) {
                        const float4 t = __ldg(reinterpret_cast<const float4*>(q + v4));
                        qs[j][v4] = t.x * p.scale; qs[j][v4 + 1] = t.y * p.scale;
                        qs[j][v4 + 2] = t.z * p.scale; qs[j][v4 + 3] = t.w * p.scale;
                    }
                } else {
                    const char* q = static_cast<const char*>(p.q) + (static_cast<size_t>(row) * p.D) * sizeof(T)
                                    + static_cast<size_t>(c) * 16;
                    float f[V];
                    Vec<T>::unpack(ldg_stream(q), f);
#pragma unroll
                    for (int v = 0; v < V; ++v) qs[j][v] = f[v] * p.scale;
                }
            }
        }
    }

    // The two butterflies below run over a lane distance that depends on the head geometry (LG lanes per head, a power of
    // two): the two common geometries (8 and 16 lanes per head) get fully unrolled instances -- as a loop with run-time bounds they cost 8 instructions
    // per step, 58 of the streaming forward's 493 per sample (ncu source page, r2 run 26).
    template <int HI, int N>                         // t[i] += over lane distances HI / 2, HI / 4, ... 1 (in this order)
    static __device__ __forceinline__ void butterfly_down(float (&t)[N]) {
#pragma unroll
        for (int off = HI >> 1; off > 0; off >>= 1) {
#pragma unroll
            for (int i = 0; i < N; ++i) t[i] += __shfl_xor_sync(FULL_MASK, t[i], off);
        }
    }
    template <int LO, int HI, int N>                 // t[i] += over lane distances LO, 2 LO, ... < HI (in this order)
    static __device__ __forceinline__ void butterfly(float (&t)[N]) {
#pragma unroll
        for (int off = LO; off < HI; off <<= 1) {
#pragma unroll
            for (int i = 0; i < N; ++i) t[i] += __shfl_xor_sync(FULL_MASK, t[i], off);
        }
    }

    // Sum x[m][j] over the lanes (and chunk columns) that make up each head.
    static __device__ __forceinline__ void head_reduce(const PoolParams& p, float (&x)[M][J]) {
        float t[M * J];
#pragma unroll
        for (int m = 0; m < M; ++m)
#pragma unroll
            for (int j = 0; j < J; ++j) t[m * J + j] = x[m][j];
        if (p.LG == 8) butterfly_down<8>(t);         // distances LG / 2 .. 1; the two common geometries unrolled
        else if (p.LG == 16) butterfly_down<16>(t);
        else {
            for (int off = p.LG >> 1; off > 0; off >>= 1) {
#pragma unroll
                for (int i = 0; i < M * J; ++i) t[i] += __shfl_xor_sync(FULL_MASK, t[i], off);
            }
        }
#pragma unroll
        for (int m = 0; m < M; ++m)
#pragma unroll
            for (int j = 0; j < J; ++j) x[m][j] = t[m * J + j];
#pragma unroll
        for (int r = 1; r < J; r <<= 1) {
            if (r < p.R) {
#pragma unroll
                for (int m = 0; m < M; ++m) {
                    float u[J];
#pragma unroll
                    for (int j = 0; j < J; ++j) u[j] = x[m][j] + x[m][j ^ r];
#pragma unroll
                    for (int j = 0; j < J; ++j) x[m][j] = u[j];
                }
            }
        }
    }

    // This warp's share of the sum over heads of x (each head of the slice counted R times).
    static __device__ __forceinline__ void head_sum_partial(const PoolParams& p, int c0, const float (&x)[M][J],
                                                            float (&part)[M]) {
#pragma unroll
        for (int m = 0; m < M; ++m) {
            float t = 0.f;
#pragma unroll
            for (int j = 0; j < J; ++j) t += in_head(p, c0, j) ? x[m][j] : 0.f;
            part[m] = t;
        }
        if (p.LG == 8) butterfly<8, 32>(part);       // distances LG .. 16; the two common geometries unrolled
        else if (p.LG == 16) butterfly<16, 32>(part);
        else {
            for (int off = p.LG; off < 32; off <<= 1) {
#pragma unroll
                for (int m = 0; m < M; ++m) part[m] += __shfl_xor_sync(FULL_MASK, part[m], off);
            }
        }
    }

    // Sum over ALL heads of the sample of x (each head counted R times; divide by H * R for the head
    // mean of torch/nn/functional.py:6657-6659).  `xchg` is a [POOL_WARPS][M] shared array; contains
    // __syncthreads() when the sample spans several warps, so every warp of the CTA must call it.
    static __device__ __forceinline__ void head_sum(const PoolParams& p, int c0, int warp, int lane,
                                                    const float (&x)[M][J], float* xchg, float (&total)[M]) {
        head_sum_partial(p, c0, x, total);
        if (p.WPS > 1) {
            if (lane == 0) {
#pragma unroll
                for (int m = 0; m < M; ++m) xchg[warp * M + m] = total[m];
            }
            __syncthreads();
            const int first = (warp / p.WPS) * p.WPS;
#pragma unroll
            for (int m = 0; m < M; ++m) {
                float t = 0.f;
                for (int s = 0; s < p.WPS; ++s) t += xchg[(first + s) * M + m];   // fixed order
                total[m] = t;
            }
            __syncthreads();                                   // xchg may be reused by the next row
        }
    }

    // Scores -> softmax -> dropout for the heads of this warp's slice.
    //   w    : softmax weights          (torch/nn/functional.py:6642-6643)
    //   wd   : post-dropout weights     (:6645)
    //   keep : dropout keep flags, bit (m * J + j); d wd / d w = keep / (1 - p)
    template <typename LoadK>
    static __device__ __forceinline__ void attention_weights(
        const PoolParams& p, const RngKey& rng, long long row, int c0, const float (&qs)[J][V], LoadK load_k,
        float (&w)[M][J], float (&wd)[M][J], unsigned& keep) {
        float s[M][J];
        key_scores(p, qs, load_k, s);
        softmax_dropout(p, rng, row, c0, s, w, wd, keep);
    }

    // head index of each of this lane's chunk columns
    static __device__ __forceinline__ void heads_of(const PoolParams& p, int c0, int (&head)[J]) {
#pragma unroll
        for (int j = 0; j < J; ++j) head[j] = min((c0 + 32 * j) >> p.logG, p.H - 1);
    }

    // Folded key projection: the scaled scores of (row, m, head) were produced by the value GEMM's side
    // output (scores = x . (scale * Wk_h^T q_h); the key bias shifts every token of a head alike and drops
    // out of the softmax).  Plain loads: 32 lanes read at most 32 / LG distinct floats of one 32-byte sector.
    static __device__ __forceinline__ void load_scores(const PoolParams& p, long long row, int c0, float (&s)[M][J]) {
        int head[J];
        heads_of(p, c0, head);
        const float* base = p.scores + static_cast<size_t>(row) * p.s_sb;
#pragma unroll
        for (int m = 0; m < M; ++m)
#pragma unroll
            for (int j = 0; j < J; ++j) s[m][j] = __ldg(base + static_cast<size_t>(m) * p.s_sm + head[j]);
    }

    // s[m][j] = (scale * q_head) . k[m, head], every lane of a head holding the head's value
    template <typename LoadK>
    static __device__ __forceinline__ void key_scores(const PoolParams& p, const float (&qs)[J][V], LoadK load_k,
                                                      float (&s)[M][J]) {
#pragma unroll
        for (int m = 0; m < M; ++m) {
            uint4 raw[J];
#pragma unroll
            for (int j = 0; j < J; ++j) raw[j] = load_k(m, j);
#pragma unroll
            for (int j = 0; j < J; ++j) {
                float f[V];
                Vec<T>::unpack(raw[j], f);
                float acc = 0.f;
#pragma unroll
                for (int v = 0; v < V; ++v) acc = fmaf(qs[j][v], f[v], acc);
                s[m][j] = acc;
            }
        }
        head_reduce(p, s);
    }

    // (+ additive mask) -> softmax over the M tokens -> dropout
    static __device__ __forceinline__ void softmax_dropout(
        const PoolParams& p, const RngKey& rng, long long row, int c0, float (&s)[M][J],
        float (&w)[M][J], float (&wd)[M][J], unsigned& keep) {
        int head[J];
        heads_of(p, c0, head);

        if (p.bias != nullptr) {                                       // :6638 baddbmm(attn_mask, q, k^T)
#pragma unroll
            for (int j = 0; j < J; ++j) {
                const float* b = p.bias + static_cast<size_t>(row) * p.bias_sb + static_cast<size_t>(head[j]) * p.bias_sh;
#pragma unroll
                for (int m = 0; m < M; ++m) s[m][j] += __ldg(b + m);
            }
        }
#pragma unroll
        for (int j = 0; j < J; ++j) {                                   // softmax over the M tokens
            float mx = s[0][j];
#pragma unroll
            for (int m = 1; m < M; ++m) mx = fmaxf(mx, s[m][j]);
            // ex2.approx / rcp: ~2^-22 relative, far inside the 1e-5 budget; the masking stage that
            // decides the mask bits keeps exact IEEE arithmetic (pool_fwd.cuh)
            float sum = 0.f;
#pragma unroll
            for (int m = 0; m < M; ++m) { w[m][j] = __expf(s[m][j] - mx); sum += w[m][j]; }
            const float inv = __frcp_rn(sum);
#pragma unroll
            for (int m = 0; m < M; ++m) w[m][j] = w[m][j] * inv;
        }
        keep = 0xffffffffu;
        if (DROP) {
            keep = 0u;
#pragma unroll
            for (int j = 0; j < J; ++j) {
#pragma unroll
                for (int blk = 0; blk < (M + 3) / 4; ++blk) {
                    float u[4];
                    draw4(rng, static_cast<unsigned long long>(row), STREAM_DROPOUT,
                          static_cast<uint32_t>(head[j]), blk, u);
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const int m = 4 * blk + i;
                        if (m < M) {
                            const bool k = (u[i] >= p.p_drop) && (p.p_drop < 1.0f);
                            keep |= k ? (1u << (m * J + j)) : 0u;
                            // w * keep / (1 - p): a true division, like the injected reference draw
                            wd[m][j] = k ? w[m][j] / p.one_minus_p : 0.f;
                        }
                    }
                }
            }
        } else {
#pragma unroll
            for (int m = 0; m < M; ++m)
#pragma unroll
                for (int j = 0; j < J; ++j) wd[m][j] = w[m][j];
        }
    }
};

// Shannon entropy with the reference's clamp: clamp(-sum xlogy(w, w), 0, log M), NaN passes through.
template <int M>
__device__ __forceinline__ float clamped_entropy(const float (&w)[M], float log_m, float* raw_out = nullptr) {
    float acc = 0.f;
#pragma unroll
    for (int m = 0; m < M; ++m)      // explicit _rn ops: never contracted to FMA, so the rounding
        acc = __fadd_rn(acc, (w[m] == 0.f) ? 0.f : __fmul_rn(w[m], logf(w[m])));   // sequence is xlogy then sum
    const float raw = -acc;
    if (raw_out) *raw_out = raw;
    return (raw != raw) ? raw : fminf(fmaxf(raw, 0.f), log_m);
}

}  // namespace aecf
