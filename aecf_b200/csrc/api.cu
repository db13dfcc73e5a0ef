// C-ABI entry points for the fused pool, plus library bookkeeping.  See include/aecf_b200.h.
#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <type_traits>

#include "pool_dispatch.cuh"

namespace aecf {

static std::atomic<unsigned long long> g_launches{0};
static thread_local char g_cuda_error[256] = "";
static thread_local char g_last_pool_kernel[128] = "";

void note_pool_kernel(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    std::vsnprintf(g_last_pool_kernel, sizeof(g_last_pool_kernel), fmt, ap);
    va_end(ap);
}

void count_launch(unsigned n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

int set_cuda_error(cudaError_t err, const char* what) {
    std::snprintf(g_cuda_error, sizeof(g_cuda_error), "%s: %s (%s)", what, cudaGetErrorName(err),
                  cudaGetErrorString(err));
    return AECF_ERR_CUDA;
}

int use_device(int device) {
    AECF_CUDA_OK(cudaSetDevice(device));
    return AECF_OK;
}

int sm_count(int device) {
    static std::atomic<int> cached[64];
    if (device < 0 || device >= 64) return 148;
    int n = cached[device].load(std::memory_order_relaxed);
    if (n == 0) {
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || n <= 0) n = 148;
        cached[device].store(n, std::memory_order_relaxed);
    }
    return n;
}

constexpr int POOL_BWD_MAX_BLOCKS = 2048;
constexpr long long POOL_BWD_CHUNK = 16;     // samples per CTA of the pool backward without batch sums (chunked schedule)

// Sum the per-block partials: d_q[D] (scaled) and d_bias_kv[2D] = [dbk | dbv].  Block (32 columns x 32
// lanes): lane y sums partials y, y+32, ... in order (all loads issued together), the 32 lane sums are
// folded in order -> deterministic.
__global__ void __launch_bounds__(1024)
pool_bwd_finalize_kernel(const float* __restrict__ partials, int blocks, int D, float scale, int q_shared,
                         float* __restrict__ d_q, float* __restrict__ d_bias_kv) {
    __shared__ float red[32][33];
    const int x = threadIdx.x & 31, y = threadIdx.x >> 5;
    const int i = blockIdx.x * 32 + x;
    float s = 0.f;
    pdl_wait();
    if (i < 3 * D && (i >= D || (q_shared && d_q))) {       // (the d_q third is not written when nobody wants it: folded)
#pragma unroll 16
        for (int b = y; b < blocks; b += 32) s += partials[static_cast<size_t>(b) * 3 * D + i];
    }
    red[y][x] = s;
    __syncthreads();
    if (y != 0 || i >= 3 * D) return;
    s = 0.f;
#pragma unroll
    for (int k = 0; k < 32; ++k) s += red[k][x];
    const int which = i / D, d = i - which * D;
    if (which == 0) { if (q_shared && d_q) d_q[d] = s * scale; }
    else if (d_bias_kv) d_bias_kv[(which == 1 ? D : 0) + d] = s;
}

struct PoolPlan {
    PoolParams p;
    MultiQuery mq;          // several queries per sample (desc.tgt_len > 1), pool_multi.cuh
    int M, J;
    bool drop, bf16, fold, multi;
    bool pad;               // padded lane map: head_dim is not a power-of-two number of 16-byte chunks (pool_core.cuh)
};

// Validate a descriptor and derive the lane/head geometry (pool_core.cuh).  `fold`: the folded-key-projection
// entry points, whose kv / scores / d_kv are matrices of B*M rows addressed by ROW strides.
static int make_plan(const aecf_pool_desc* d, PoolPlan* plan, bool fold = false) {
    if (d == nullptr) return AECF_ERR_INVALID;
    if (d->batch < 0 || d->embed_dim <= 0 || d->num_heads <= 0 || d->num_tokens <= 0) return AECF_ERR_INVALID;
    if (d->embed_dim % d->num_heads != 0) return AECF_ERR_INVALID;
    if (d->dtype != AECF_F32 && d->dtype != AECF_BF16) return AECF_ERR_INVALID;
    if (d->offset >> 32) return AECF_ERR_INVALID;
    if (!(d->dropout_p >= 0.f && d->dropout_p <= 1.f)) return AECF_ERR_INVALID;
    if (d->masking < 0 || d->masking > 2) return AECF_ERR_INVALID;
    if (d->num_tokens > AECF_MAX_TOKENS) return AECF_ERR_UNSUPPORTED;
    const int V = d->dtype == AECF_BF16 ? 8 : 4;
    const int D = d->embed_dim, H = d->num_heads, hd = D / H;
    if (hd % V != 0) return AECF_ERR_UNSUPPORTED;
    const int GR = hd / V;                           // real chunks per head
    const int G = 1 << ilog2(GR);                    // the head's span in the lane map: GR, or padded to a power of two
    const int NC = D / V;
    const int NCV = H * G;                           // chunks of the lane map's row (NC unless padded)
    // J chunk columns per lane: enough to hold a whole head in one warp (R <= J), and two columns
    // (512 contiguous bytes x 2 per token) whenever the row is long enough.
    const int R = G < 32 ? 1 : G / 32;
    int J = NCV > 32 ? 2 : 1;
    if (J < R) J = R;
    if (J > 4) return AECF_ERR_UNSUPPORTED;          // head_dim > 128 * V elements
    int WPS = (NCV + 32 * J - 1) / (32 * J);
    // a row must split over a power-of-two number of warps: rows of 3 * 2^k slices (D = 768 in fp32, 1536 in bf16)
    // take wider slices instead, whose last warp is then partly idle
    while ((WPS > POOL_WARPS || !is_pow2(WPS)) && J < 4) {
        J *= 2;
        WPS = (NCV + 32 * J - 1) / (32 * J);
    }
    if (WPS > POOL_WARPS || !is_pow2(WPS)) return AECF_ERR_UNSUPPORTED;

    PoolParams& p = plan->p;
    std::memset(&p, 0, sizeof(p));
    p.B = d->batch; p.D = D; p.H = H; p.NC = NC; p.G = G; p.logG = ilog2(G);
    p.LG = G < 32 ? G : 32; p.R = R; p.WPS = WPS; p.SPC = POOL_WARPS / WPS;
    p.GR = GR;
    p.scale = static_cast<float>(std::sqrt(1.0 / static_cast<double>(hd)));   // math.sqrt(1.0 / float(E)), functional.py:6632
    p.p_drop = d->dropout_p;
    p.one_minus_p = static_cast<float>(1.0 - static_cast<double>(d->dropout_p));
    p.base_mask_prob = d->base_mask_prob;
    p.log_m = static_cast<float>(std::log(static_cast<double>(d->num_tokens)));   // math.log(seq_len), AECFLayer.py:127,191
    p.training = d->training; p.masking = d->masking; p.min_active = d->min_active;
    p.q_shared = d->q_is_shared;
    p.rng.k0 = static_cast<uint32_t>(d->seed); p.rng.k1 = static_cast<uint32_t>(d->seed >> 32);
    p.rng.offset = static_cast<uint32_t>(d->offset); p.rng.row0 = d->row0;
    p.rng_state = reinterpret_cast<const unsigned long long*>(d->rng_state);
    p.bias_sb = d->bias_stride_b; p.bias_sh = d->bias_stride_h;
    if (fold) {
        if (!d->q_is_shared) return AECF_ERR_UNSUPPORTED;       // the fold needs one query for all rows
        long long rs_b = d->kv_stride_b, rs_m = d->kv_stride_m;   // in rows of the [B*M, .] matrices
        if (rs_b == 0 && rs_m == 0) { rs_b = d->num_tokens; rs_m = 1; }
        if (rs_b < 1 || rs_m < 1) return AECF_ERR_INVALID;
        const int hsp = aecf_fold_score_cols(d->dtype, H);
        p.HSP = hsp;
        p.kv_sb = rs_b * D; p.kv_sm = rs_m * D;
        p.dkv_sb = rs_b * (D + hsp); p.dkv_sm = rs_m * (D + hsp);
        const int hs = (H + 3) & ~3;
        p.s_sb = rs_b * hs; p.s_sm = rs_m * hs;
    } else if (d->kv_stride_b == 0 && d->kv_stride_m == 0) {
        p.kv_sm = 2LL * D; p.kv_sb = p.kv_sm * d->num_tokens;
        p.dkv_sb = p.kv_sb; p.dkv_sm = p.kv_sm;
    } else {
        if (d->kv_stride_b < 2LL * D || d->kv_stride_m < 2LL * D) return AECF_ERR_INVALID;
        if ((d->kv_stride_b * (16 / V)) % 16 != 0 || (d->kv_stride_m * (16 / V)) % 16 != 0) return AECF_ERR_ALIGNMENT;
        p.kv_sb = d->kv_stride_b; p.kv_sm = d->kv_stride_m;
        p.dkv_sb = p.kv_sb; p.dkv_sm = p.kv_sm;
    }
    const int S = d->tgt_len > 1 ? d->tgt_len : 1;
    plan->multi = S > 1;
    std::memset(&plan->mq, 0, sizeof(plan->mq));
    if (plan->multi) {
        if (fold || d->q_is_shared) return AECF_ERR_UNSUPPORTED;    // per-row queries, unfolded key projection
        long long rb = d->q_stride_b, rs = d->q_stride_s;
        if (rb == 0 && rs == 0) { rb = S; rs = 1; }                 // batch-first [B, S, D]
        if (rb < 1 || rs < 1 || d->bias_stride_s < 0) return AECF_ERR_INVALID;
        if (d->batch > (1LL << 40) / S) return AECF_ERR_INVALID;
        plan->mq.S = S; plan->mq.q_rb = rb; plan->mq.q_rs = rs;
        plan->mq.bias_sb = d->bias_stride_b; plan->mq.bias_sh = d->bias_stride_h; plan->mq.bias_ss = d->bias_stride_s;
        p.rng.row0 = d->row0 * static_cast<unsigned long long>(S);  // Philox row of (b, s): (row0 + b) * S + s
    }
    if (d->row_index != nullptr) {
        if (!d->q_is_shared || plan->multi) return AECF_ERR_UNSUPPORTED;
        if (d->src_rows < d->batch) return AECF_ERR_INVALID;
        if (p.bias_sb != 0 || p.bias_sh != 0) return AECF_ERR_UNSUPPORTED;      // a per-row score bias would need the indirection too
        p.row_index = reinterpret_cast<const long long*>(d->row_index);
    }
    plan->fold = fold;
    plan->M = d->num_tokens; plan->J = J;
    plan->drop = d->training && d->dropout_p > 0.f;
    plan->bf16 = d->dtype == AECF_BF16;
    plan->pad = GR != G;
    return AECF_OK;
}

// Calls f(T{}, DROP, PAD) with the plan's element type and the std::bool_constant of its dropout and lane map: the
// instantiation set of pool_dispatch.cuh that the plan runs.
template <typename F>
static int with_pool_types(const PoolPlan& plan, F&& f) {
    auto pad = [&](auto t, auto drop) { return plan.pad ? f(t, drop, std::true_type{}) : f(t, drop, std::false_type{}); };
    auto drop = [&](auto t) { return plan.drop ? pad(t, std::true_type{}) : pad(t, std::false_type{}); };
    return plan.bf16 ? drop(__nv_bfloat16{}) : drop(float{});
}

}  // namespace aecf

using namespace aecf;

extern "C" {

int aecf_abi_version(void) { return AECF_ABI_VERSION; }

const char* aecf_strerror(int status) {
    switch (status) {
        case AECF_OK: return "ok";
        case AECF_ERR_INVALID: return "invalid argument";
        case AECF_ERR_UNSUPPORTED: return "shape or dtype outside what the sm_100a kernels cover (no fallback by design)";
        case AECF_ERR_ALIGNMENT: return "pointer or leading dimension not 16-byte aligned";
        case AECF_ERR_WORKSPACE: return "workspace too small";
        case AECF_ERR_CUDA: return "CUDA error (see aecf_last_cuda_error)";
        default: return "unknown status";
    }
}

const char* aecf_last_cuda_error(void) { return g_cuda_error; }
const char* aecf_pool_last_kernel(void) { return g_last_pool_kernel; }
uint64_t aecf_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }
const char* aecf_build_info(void) {
    return "aecf_b200 abi " AECF_STR(AECF_ABI_VERSION) ", sm_100a, nvcc " AECF_STR(__CUDACC_VER_MAJOR__) "." AECF_STR(__CUDACC_VER_MINOR__);
}

}  // extern "C"

// the streaming forward kernel (one warp per sample, at most one CTA per SM) carries the fused entropy_loss term
static bool pool_fwd_carries_loss(const PoolPlan& plan, const aecf_pool_desc& d) {
    return !plan.multi && plan.p.WPS == 1 && d.masking == 1 && d.row_index == nullptr && sm_count(d.device) <= POOL_LOSS_MAX_CTAS;
}

static int pool_fwd_impl(const aecf_pool_desc* desc, bool fold, const void* q, const float* scores, const void* kv,
                         const float* score_bias, void* ctx, float* pooled, float* entropy, float* mask_rate,
                         float* masked, uint8_t* mask_bits, void* stream) {
    PoolPlan plan;
    int rc = make_plan(desc, &plan, fold);
    if (rc != AECF_OK) return rc;
    if (desc->batch == 0) return AECF_OK;
    if ((!fold && !q) || (fold && !scores) || !kv || !ctx || !pooled) return AECF_ERR_INVALID;
    if ((q && !aligned16(q)) || !aligned16(kv) || !aligned16(ctx)) return AECF_ERR_ALIGNMENT;
    if (desc->row_index != nullptr && score_bias != nullptr) return AECF_ERR_UNSUPPORTED;
    DeviceScope device_scope__(desc->device);
    if ((rc = device_scope__.rc) != AECF_OK) return rc;
    PoolParams& p = plan.p;
    p.q = q; p.kv = kv; p.bias = score_bias; p.scores = scores;
    p.ctx = ctx; p.pooled = pooled; p.entropy = entropy; p.mask_rate = mask_rate; p.masked = masked;
    p.mask_bits = mask_bits;
    const int sms = sm_count(desc->device);
    if (desc->loss_out != nullptr && pool_fwd_carries_loss(plan, *desc)) {
        if (desc->loss_workspace == nullptr || !aligned16(desc->loss_workspace)) return AECF_ERR_INVALID;
        p.loss_out = desc->loss_out;
        p.loss_partials = static_cast<float*>(desc->loss_workspace);
        p.loss_ticket = reinterpret_cast<unsigned*>(p.loss_partials + POOL_LOSS_MAX_CTAS);
        p.loss_target = desc->loss_target;
    }
    TimedLaunch timed(static_cast<cudaStream_t>(stream));
    if (plan.multi) {                                   // one warp slice per (b, s) row; the bias travels in mq
        plan.mq.bias = score_bias;
        p.bias = nullptr;
        const int rows_grid = static_cast<int>((p.B * plan.mq.S + p.SPC - 1) / p.SPC);
        note_pool_kernel("multi fwd M=%d J=%d PAD=%d grid=%d", plan.M, plan.J, int(plan.pad), rows_grid);
        return with_pool_types(plan, [&](auto t, auto drop, auto pad) {
            return launch_pool_fwd_multi<decltype(t), drop, pad>(plan.M, plan.J, p, plan.mq, rows_grid, stream);
        });
    }
    const int grid = static_cast<int>((p.B + p.SPC - 1) / p.SPC);
    return with_pool_types(plan, [&](auto t, auto drop, auto pad) {
        return launch_pool_fwd<decltype(t), drop, pad>(plan.M, plan.J, p, grid, sms, fold, stream);
    });
}

extern "C" {

int aecf_fold_score_cols(int32_t dtype, int32_t num_heads) {
    const int per16 = dtype == AECF_BF16 ? 8 : 4;
    return (num_heads + per16 - 1) / per16 * per16;
}

int aecf_pool_fwd(const aecf_pool_desc* desc, const void* q, const void* kv, const float* score_bias,
                  void* ctx, float* pooled, float* entropy, float* mask_rate, float* masked,
                  uint8_t* mask_bits, void* stream) {
    return pool_fwd_impl(desc, false, q, nullptr, kv, score_bias, ctx, pooled, entropy, mask_rate, masked, mask_bits, stream);
}

size_t aecf_pool_loss_workspace_bytes(void) { return POOL_LOSS_MAX_CTAS * sizeof(float) + 64; }

int aecf_pool_fwd_has_loss(const aecf_pool_desc* desc, int32_t folded) {
    PoolPlan plan;
    if (make_plan(desc, &plan, folded != 0) != AECF_OK) return 0;
    return pool_fwd_carries_loss(plan, *desc) ? 1 : 0;
}

int aecf_pool_fwd_folded(const aecf_pool_desc* desc, const float* scores, const void* v, const float* score_bias,
                         void* ctx, float* pooled, float* entropy, float* mask_rate, float* masked,
                         uint8_t* mask_bits, void* stream) {
    return pool_fwd_impl(desc, true, nullptr, scores, v, score_bias, ctx, pooled, entropy, mask_rate, masked, mask_bits, stream);
}

size_t aecf_pool_bwd_workspace_bytes(const aecf_pool_desc* desc) {
    if (desc == nullptr || desc->embed_dim <= 0) return 0;
    return static_cast<size_t>(POOL_BWD_MAX_BLOCKS) * 3 * desc->embed_dim * sizeof(float);
}

}  // extern "C"

static int pool_bwd_impl(const aecf_pool_desc* desc, bool fold, const void* q, const float* scores, const void* kv,
                         const float* score_bias, const void* d_ctx, const float* d_pooled, const float* d_entropy,
                         void* d_kv, void* d_q, float* d_bias_kv, void* workspace, size_t workspace_bytes, void* stream,
                         bool no_sums = false, float* rowsum = nullptr) {
    PoolPlan plan;
    int rc = make_plan(desc, &plan, fold);
    if (rc != AECF_OK) return rc;
    if (!q || !kv || !d_ctx || !d_kv || (!fold && !d_q) || (fold && !scores) || (!workspace && !no_sums)) return AECF_ERR_INVALID;
    if (!aligned16(q) || !aligned16(kv) || !aligned16(d_ctx) || !aligned16(d_kv) || (d_q && !aligned16(d_q)) ||
        !aligned16(workspace))
        return AECF_ERR_ALIGNMENT;
    if (!no_sums && workspace_bytes < aecf_pool_bwd_workspace_bytes(desc)) return AECF_ERR_WORKSPACE;
    if (no_sums && (!fold || plan.multi)) return AECF_ERR_INVALID;
    if (desc->row_index != nullptr && score_bias != nullptr) return AECF_ERR_UNSUPPORTED;
    if (desc->batch == 0) return AECF_OK;
    DeviceScope device_scope__(desc->device);
    if ((rc = device_scope__.rc) != AECF_OK) return rc;
    PoolParams& p = plan.p;
    p.q = q; p.kv = kv; p.bias = score_bias; p.scores = scores;
    p.d_ctx = d_ctx; p.d_pooled = d_pooled; p.d_entropy = d_entropy; p.d_kv = d_kv; p.d_q = d_q;
    p.partials = no_sums ? nullptr : static_cast<float*>(workspace);
    p.rowsum = no_sums ? rowsum : nullptr;

    int per_sm = 1;                                     // pool_bwd_multi_kernel: __launch_bounds__(256, 1)
    if (!plan.multi)
        per_sm = with_pool_types(plan, [&](auto t, auto drop, auto pad) {
            return pool_bwd_blocks_per_sm<decltype(t), drop, pad>(plan.M, plan.J, fold);
        });
    if (per_sm <= 0) per_sm = 1;
    long long want = (p.B + p.SPC - 1) / p.SPC;
    long long cap = static_cast<long long>(sm_count(desc->device)) * per_sm;   // persistent: one resident wave
    if (cap > POOL_BWD_MAX_BLOCKS) cap = POOL_BWD_MAX_BLOCKS;
    int grid = static_cast<int>(want < cap ? want : cap);
    if (grid < 1) grid = 1;
    // Chunked schedule (pool_bwd.cuh), for the kernel without batch sums: CTA b owns `chunk` consecutive samples, several
    // CTAs per resident slot, handed out by the block scheduler as CTAs retire.  POOL_BWD_CHUNK samples per CTA, rounded
    // up to whole slices of SPC samples and doubled until the grid fits in an int.
    if (no_sums) {
        long long chunk = (POOL_BWD_CHUNK + p.SPC - 1) / p.SPC * p.SPC;
        while ((p.B + chunk - 1) / chunk > 0x7fffffffLL) chunk *= 2;
        p.chunk = chunk;
        grid = static_cast<int>((p.B + chunk - 1) / chunk);
        note_pool_kernel("bwd chunked M=%d J=%d PAD=%d fold=%d grid=%d chunk=%lld", plan.M, plan.J, int(plan.pad), int(fold),
                         grid, chunk);
    } else {                                            // passes: slices of SPC samples per CTA, the last pass partial
        note_pool_kernel("%s M=%d J=%d PAD=%d fold=%d grid=%d passes=%lld", plan.multi ? "multi bwd" : "bwd grid-stride",
                         plan.M, plan.J, int(plan.pad), int(fold), grid, (want + grid - 1) / grid);
    }

    {
        TimedLaunch timed(static_cast<cudaStream_t>(stream));
        if (plan.multi) {
            plan.mq.bias = score_bias;
            p.bias = nullptr;
        }
        rc = with_pool_types(plan, [&](auto t, auto drop, auto pad) {
            return plan.multi ? launch_pool_bwd_multi<decltype(t), drop, pad>(plan.M, plan.J, p, plan.mq, grid, stream)
                              : launch_pool_bwd<decltype(t), drop, pad>(plan.M, plan.J, p, grid, fold, stream);
        });
    }
    if (rc != AECF_OK) return rc;
    if (no_sums) return AECF_OK;                        // the caller forms the batch sums itself (grad_tail.cu)
    const int n = 3 * p.D;
    TimedLaunch timed_finalize(static_cast<cudaStream_t>(stream), AECF_SITE_POOL_BWD_FINALIZE);
    AECF_CUDA_OK(launch_pdl(pool_bwd_finalize_kernel, dim3((n + 31) / 32), dim3(1024), 0, static_cast<cudaStream_t>(stream),
                            p.partials, grid, p.D, p.scale, p.q_shared, p.q_shared ? static_cast<float*>(d_q) : nullptr,
                            d_bias_kv));
    count_launch();
    return AECF_OK;
}

namespace aecf {
// fusion.cu: the folded backward without its batch sums (pool_bwd.cuh).  rowsum null: nothing is left for the tail to sum
// (no dropout, every sample pooled); else the kernel leaves [s | sum_m ds] per sample and head there ([src_rows][2 HSP] fp32).
int pool_bwd_folded_nosums(const aecf_pool_desc* desc, const void* q_proj, const float* scores, const void* v,
                           const float* score_bias, const void* d_ctx, const float* d_pooled, const float* d_entropy,
                           void* d_vs, float* rowsum, void* stream) {
    return pool_bwd_impl(desc, true, q_proj, scores, v, score_bias, d_ctx, d_pooled, d_entropy, d_vs, nullptr, nullptr,
                         nullptr, 0, stream, true, rowsum);
}
}  // namespace aecf

extern "C" {

int aecf_pool_bwd(const aecf_pool_desc* desc, const void* q, const void* kv, const float* score_bias,
                  const void* d_ctx, const float* d_pooled, const float* d_entropy,
                  void* d_kv, void* d_q, float* d_bias_kv,
                  void* workspace, size_t workspace_bytes, void* stream) {
    return pool_bwd_impl(desc, false, q, nullptr, kv, score_bias, d_ctx, d_pooled, d_entropy, d_kv, d_q, d_bias_kv,
                         workspace, workspace_bytes, stream);
}

int aecf_pool_bwd_folded(const aecf_pool_desc* desc, const void* q_proj, const float* scores, const void* v,
                         const float* score_bias, const void* d_ctx, const float* d_pooled, const float* d_entropy,
                         void* d_vs, float* d_bias_kv, void* workspace, size_t workspace_bytes, void* stream) {
    return pool_bwd_impl(desc, true, q_proj, scores, v, score_bias, d_ctx, d_pooled, d_entropy, d_vs, nullptr, d_bias_kv,
                         workspace, workspace_bytes, stream);
}

}  // extern "C"
