// Whole-step entry points: the complete MultimodalAttentionPool forward / backward as one C-ABI call
// each (include/aecf_b200.h).  They compose the per-kernel entry points in the order the reference's
// call chain implies (reference aecf/AECFLayer.py:515-541 over torch/nn/functional.py:5847-5865,
// 6630-6659; backward per SURVEY.md Appendix B), so the host pays one FFI crossing per direction.
#include "common.cuh"
#include "grad_tail.cuh"

namespace aecf {

// [d_qp fp32 D | d_bias_kv fp32 2D] -> in_proj_bias gradient [3D] in the gradient dtype
template <typename T>
__global__ void pack_in_bias_kernel(const float* __restrict__ d_q, const float* __restrict__ d_bias_kv, int D,
                                    T* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    pdl_wait();
    if (i >= 3 * D) return;
    out[i] = from_float<T>(i < D ? d_q[i] : d_bias_kv[i - D]);
}

struct Geometry {
    long long B, rows, QR;     // samples, key/value rows (B * M), query rows (B * S)
    int M, D, H, es, dt;
    int gdt, ges;      // dtype and element size of the parameter gradients (fp32 in mixed precision, else dt)
    bool shared, fold;
    int HS, HSP;       // folded key projection: score columns (fp32, H rounded up to 4) / score-gradient columns (dt, 16-byte multiple)
};

static int geometry(const aecf_pool_desc* d, Geometry* g) {
    if (!d || d->batch < 0 || d->embed_dim <= 0 || d->num_tokens <= 0) return AECF_ERR_INVALID;
    if (d->dtype != AECF_F32 && d->dtype != AECF_BF16) return AECF_ERR_INVALID;
    if (d->param_grads_f32 != 0 && (d->param_grads_f32 != 1 || d->dtype != AECF_BF16)) return AECF_ERR_INVALID;
    g->B = d->batch; g->M = d->num_tokens; g->D = d->embed_dim;
    // row indirection: the pool kernels take the `batch` listed rows, the products around them all `src_rows` samples
    const long long samples = d->row_index != nullptr ? d->src_rows : d->batch;
    if (d->row_index != nullptr && (d->src_rows < d->batch || d->tgt_len > 1 || !d->q_is_shared)) return AECF_ERR_UNSUPPORTED;
    g->rows = samples * g->M;
    g->QR = samples * (d->tgt_len > 1 ? d->tgt_len : 1);
    g->dt = d->dtype; g->es = d->dtype == AECF_BF16 ? 2 : 4; g->shared = d->q_is_shared != 0;
    g->gdt = d->param_grads_f32 ? AECF_F32 : d->dtype; g->ges = g->gdt == AECF_BF16 ? 2 : 4;
    g->H = d->num_heads; g->fold = d->fold_key != 0;
    g->HS = (g->H + 3) & ~3; g->HSP = aecf_fold_score_cols(d->dtype, g->H);
    if (g->fold && (!g->shared || g->H <= 0 || g->H > 32)) return AECF_ERR_UNSUPPORTED;
    if (d->tgt_len > 1 && (g->shared || g->fold)) return AECF_ERR_UNSUPPORTED;   // several queries per sample: per-row, unfolded
    return AECF_OK;
}

static const void* at(const void* p, long long elems, int es) {
    return p ? static_cast<const char*>(p) + elems * es : nullptr;
}
static void* at(void* p, long long elems, int es) { return p ? static_cast<char*>(p) + elems * es : nullptr; }

// api.cu
int pool_bwd_folded_nosums(const aecf_pool_desc* desc, const void* q_proj, const float* scores, const void* v,
                           const float* score_bias, const void* d_ctx, const float* d_pooled, const float* d_entropy,
                           void* d_vs, float* rowsum, void* stream);

struct Workspace {
    char* gemm; size_t gemm_bytes;
    char* pool; size_t pool_bytes;
    char* colsum; size_t colsum_bytes;
    float* d_qp;       // [D]
    float* d_bias_kv;  // [2D]
    float* d_bq;       // [D] (per-row query)
    // folded backward with the fused gradient tail (grad_tail.cu): the two weight-gradient products leave their split-K
    // partials side by side, then the raw sums and the tail's scratch
    char* gemm_o; size_t gemm_o_bytes;
    char* gemm_g; size_t gemm_g_bytes;
    float* sums;
    char* tail; size_t tail_bytes;
    float* rowsum; size_t rowsum_bytes;   // [samples][2 HSP] fp32: what the pool backward leaves for the tail's bias sums
    size_t total;
};

#define AECF_TRY(expr)                   \
    do {                                 \
        const int rc__ = (expr);         \
        if (rc__ != AECF_OK) return rc__; \
    } while (0)

static size_t align256(size_t x) { return (x + 255) & ~static_cast<size_t>(255); }

static aecf_gemm_desc gemm_desc(int device, int dta, int dtb, int dtc, int dtbias, int al, int bl, long long m,
                                long long n, long long k, long long lda, long long ldb, long long ldc) {
    aecf_gemm_desc g{};
    g.device = device; g.dtype_a = dta; g.dtype_b = dtb; g.dtype_c = dtc; g.dtype_bias = dtbias;
    g.a_layout = al; g.b_layout = bl; g.accumulate = 0; g.impl = AECF_GEMM_AUTO;
    g.m = m; g.n = n; g.k = k; g.lda = lda; g.ldb = ldb; g.ldc = ldc;
    return g;
}

// Largest GEMM workspace any product of the step can ask for (split-K partials of the weight gradients).
static size_t max_gemm_workspace(const aecf_pool_desc* d, const Geometry& g) {
    const int dt = g.dt, gdt = g.gdt, D = g.D;
    size_t need = 16;
    const aecf_gemm_desc probes[] = {
        gemm_desc(d->device, dt, dt, gdt, dt, AECF_MN_MAJOR, AECF_MN_MAJOR, 2 * D, D, g.rows, 2 * D, D, D),  // dW_kv
        gemm_desc(d->device, dt, dt, gdt, dt, AECF_MN_MAJOR, AECF_MN_MAJOR, D, D, g.rows, 2 * D, D, D),      // dW_k / dW_v
        gemm_desc(d->device, dt, dt, gdt, dt, AECF_MN_MAJOR, AECF_MN_MAJOR, D, D, g.QR, D, D, D),            // dW_o, dW_q
        gemm_desc(d->device, dt, dt, dt, dt, AECF_K_MAJOR, AECF_K_MAJOR, g.rows, 2 * D, D, D, D, 2 * D),     // kv
        gemm_desc(d->device, dt, dt, dt, dt, AECF_K_MAJOR, AECF_MN_MAJOR, g.rows, D, 2 * D, 2 * D, D, D),    // dX
        gemm_desc(d->device, dt, dt, AECF_F32, dt, AECF_MN_MAJOR, AECF_MN_MAJOR, D + g.HSP, D, g.rows, D + g.HSP, D, D),   // folded [dWv ; R]
        gemm_desc(d->device, dt, dt, dt, dt, AECF_K_MAJOR, AECF_MN_MAJOR, g.rows, D, D + g.HSP, D + g.HSP, D, D),          // folded dX
        gemm_desc(d->device, dt, dt, dt, dt, AECF_K_MAJOR, AECF_K_MAJOR, g.rows, D, D, D, D, D),                           // folded V
        // the [query rows, D] x [D, D] products: per-row q_proj, out_proj / d_ctx, d_query (split-K at D = 2048, small batch)
        gemm_desc(d->device, dt, dt, dt, dt, AECF_K_MAJOR, AECF_K_MAJOR, g.QR, D, D, D, D, D),
        gemm_desc(d->device, dt, dt, dt, dt, AECF_K_MAJOR, AECF_MN_MAJOR, g.QR, D, D, D, D, D),
        gemm_desc(d->device, dt, dt, AECF_F32, dt, AECF_K_MAJOR, AECF_K_MAJOR, 1, D, D, D, D, D),                          // shared query
    };
    for (const aecf_gemm_desc& p : probes) {
        const size_t w = aecf_gemm_workspace_bytes(&p);
        if (w > need) need = w;
    }
    return need;
}

static int carve(const aecf_pool_desc* d, const Geometry& g, void* base, Workspace* w) {
    w->gemm_bytes = align256(max_gemm_workspace(d, g));
    w->pool_bytes = align256(aecf_pool_bwd_workspace_bytes(d));
    w->colsum_bytes = align256(aecf_colsum_workspace_bytes(g.QR, g.D));
    size_t off = 0;
    char* b = static_cast<char*>(base);
    w->gemm = b + off; off += w->gemm_bytes;
    w->pool = b + off; off += w->pool_bytes;
    w->colsum = b + off; off += w->colsum_bytes;
    w->d_qp = reinterpret_cast<float*>(b + off); off += align256(sizeof(float) * g.D);
    w->d_bias_kv = reinterpret_cast<float*>(b + off); off += align256(sizeof(float) * 2 * g.D);
    w->d_bq = reinterpret_cast<float*>(b + off); off += align256(sizeof(float) * g.D);
    w->gemm_o = w->gemm_g = w->tail = nullptr; w->sums = nullptr; w->rowsum = nullptr;
    w->gemm_o_bytes = w->gemm_g_bytes = w->tail_bytes = w->rowsum_bytes = 0;
    if (g.fold) {
        const int dt = g.dt, D = g.D, KF = g.D + g.HSP;
        const aecf_gemm_desc o = gemm_desc(d->device, dt, dt, AECF_F32, dt, AECF_MN_MAJOR, AECF_MN_MAJOR, D, D, g.QR, D, D, D);
        const aecf_gemm_desc kv = gemm_desc(d->device, dt, dt, AECF_F32, dt, AECF_MN_MAJOR, AECF_MN_MAJOR, KF, D, g.rows, KF, D, D);
        w->gemm_o_bytes = align256(gemm_partials_workspace_bytes(&o));
        w->gemm_g_bytes = align256(gemm_partials_workspace_bytes(&kv));
        w->tail_bytes = align256(grad_tail_scratch_bytes(D, sm_count(d->device)));
        w->gemm_o = b + off; off += w->gemm_o_bytes;
        w->gemm_g = b + off; off += w->gemm_g_bytes;
        w->sums = reinterpret_cast<float*>(b + off); off += align256(sizeof(float) * tail_layout(D, g.HSP).total);
        w->tail = b + off; off += w->tail_bytes;
        w->rowsum_bytes = align256(sizeof(float) * 2 * g.HSP * static_cast<size_t>(g.QR));
        w->rowsum = reinterpret_cast<float*>(b + off); off += w->rowsum_bytes;
    }
    w->total = off;
    return AECF_OK;
}

// ---- the folded backward: five launches on `s`, the gradient tail next to them ----
//   s    : dWo partials -> d_ctx -> pool backward -(fork)-> [dWv ; R] partials -(fork 2)-> dX -(join)->
//   side :                                          colsum(d_out), dWo fold,  [dWv ; R] fold, partial folds -> [peer sum] -> finish
//                                                   bias sums over d_ctx
// Each half of the tail runs next to a tensor-core product that leaves half of the HBM bandwidth unused.
static int folded_backward(const aecf_pool_desc* desc, const Geometry& g, const aecf_fusion_tensors* t,
                           const aecf_fusion_grads* gr, const Workspace& w, cudaStream_t s) {
    const int dt = g.dt, D = g.D, dev = desc->device, KF = g.D + g.HSP;
    const bool want_in = gr->d_in_proj_weight || gr->d_query || gr->d_in_proj_bias;
    const bool want_tail = want_in || gr->d_out_proj_weight || gr->d_out_proj_bias;
    const aecf_dp_desc* dp = (gr->dp != nullptr && gr->dp->world > 1) ? gr->dp : nullptr;
    if (dp != nullptr && (dp->rank < 0 || dp->rank >= dp->world || dp->world > 8 || !dp->sums || !dp->reduced || !dp->flags))
        return AECF_ERR_INVALID;
    const bool forked = gr->side_stream != nullptr && gr->fork_event != nullptr && gr->fork_event2 != nullptr &&
                        gr->join_event != nullptr && want_tail;
    cudaStream_t side = forked ? static_cast<cudaStream_t>(gr->side_stream) : s;
    GradTailArgs a{};
    a.dtype = dt; a.grad_dtype = g.gdt; a.D = D; a.H = g.H; a.HSP = g.HSP; a.sms = sm_count(dev);
    a.scratch = w.tail;
    a.sums = dp ? static_cast<float*>(dp->sums[dp->rank]) : w.sums;
    a.q_proj = static_cast<const float*>(t->q_proj); a.in_proj_weight = t->in_proj_weight; a.query = t->query;
    a.d_in_w = gr->d_in_proj_weight; a.d_in_b = gr->d_in_proj_bias; a.d_out_w = gr->d_out_proj_weight;
    a.d_out_b = gr->d_out_proj_bias; a.d_query = gr->d_query;
    a.d_out = (gr->d_out_proj_bias || gr->d_in_proj_bias) ? gr->d_out : nullptr; a.rows = g.QR;   // (the in-projection bias may need the sums too)

    if (gr->d_out_proj_weight) {                             // dWo = g^T ctx, left as split-K partials
        ScopedSite site(AECF_SITE_D_OUT_WEIGHT);
        const aecf_gemm_desc d = gemm_desc(dev, dt, dt, AECF_F32, dt, AECF_MN_MAJOR, AECF_MN_MAJOR, D, D, g.QR, D, D, D);
        AECF_TRY(gemm_partials(&d, gr->d_out, t->ctx, w.gemm_o, w.gemm_o_bytes, s, &a.o));
    }
    {                                                        // d_ctx = g Wo
        ScopedSite site(AECF_SITE_D_CTX);
        const aecf_gemm_desc d = gemm_desc(dev, dt, dt, dt, dt, AECF_K_MAJOR, AECF_MN_MAJOR, g.QR, D, D, D, D, D);
        AECF_TRY(aecf_gemm(&d, gr->d_out, t->out_proj_weight, nullptr, gr->d_ctx, w.gemm, w.gemm_bytes, s));
    }
    // The value and key thirds of the in-projection bias gradient (pool_bwd.cuh).  No dropout, no mask, every sample pooled:
    // the softmax weights of a sample sum to one, so d_bias_v = sum_b d_ctx[b, :] = Wo^T colsum(d_out) and d_bias_k = 0 -- the
    // tail forms them from the column sums of d_out and the pool backward carries no batch sums at all.  Otherwise the kernel
    // leaves [s | sum_m ds] per sample and head and the tail walks d_ctx once more.  A mask can cover every token of a
    // sample: its weights are then NaN, not summing to one, and these sums are NaN as in torch.
    const bool bias_from_bo = desc->row_index == nullptr && t->score_bias == nullptr && !(desc->training && desc->dropout_p > 0.f);
    float* rowsum = (gr->d_in_proj_bias && !bias_from_bo) ? w.rowsum : nullptr;
    if (desc->row_index != nullptr) {                            // unlisted samples: zero rows of [dV | ds], no share in the bias sums
        AECF_CUDA_OK(cudaMemsetAsync(gr->d_kv, 0, static_cast<size_t>(g.rows) * KF * g.es, s));
        if (rowsum) AECF_CUDA_OK(cudaMemsetAsync(rowsum, 0, w.rowsum_bytes, s));
    }
    {
        ScopedSite site(AECF_SITE_POOL_BWD);
        AECF_TRY(pool_bwd_folded_nosums(desc, t->q_proj, t->scores, t->kv, t->score_bias, gr->d_ctx, gr->d_pooled,
                                        gr->d_entropy, gr->d_kv, rowsum, s));
        if (rowsum) { a.rowsum = rowsum; a.d_ctx = gr->d_ctx; a.samples = g.QR; }
        else if (gr->d_in_proj_bias) a.out_proj_weight = t->out_proj_weight;      // d_bias_v = Wo^T colsum(d_out)
    }
    // Each half of the tail is enqueued AFTER the product it runs next to: the product's persistent CTAs (one per SM, all
    // but 2 KB of its shared memory) are placed first and the tail's blocks fill in beside them -- the other way round a
    // product CTA finds its SM taken and the whole product ends late by as long as it waited.
    if (forked) AECF_CUDA_OK(cudaEventRecord(static_cast<cudaEvent_t>(gr->fork_event), s));          // after the pool backward
    if (want_in) {                                           // [dWv ; R] = [dV | ds]^T X, left as split-K partials
        ScopedSite site(AECF_SITE_D_KV_WEIGHT);
        const aecf_gemm_desc d = gemm_desc(dev, dt, dt, AECF_F32, dt, AECF_MN_MAJOR, AECF_MN_MAJOR, KF, D, g.rows, KF, D, D);
        AECF_TRY(gemm_partials(&d, gr->d_kv, t->key, w.gemm_g, w.gemm_g_bytes, s, &a.g));
    }
    if (want_tail) {
        // first half of the tail (column sums of d_out, dWo fold: 86 MB of reads at config 2) next to the [dWv ; R] product.
        // Not earlier: next to the pool backward it would only take HBM bandwidth from a kernel that is bound by it
        // (r2 run 5: pool_bwd 88 -> 131 us), and the d_ctx product's CTAs leave no shared memory for a second CTA.
        if (forked) AECF_CUDA_OK(cudaStreamWaitEvent(side, static_cast<cudaEvent_t>(gr->fork_event), 0));
        AECF_TRY(launch_grad_gather(a, GATHER_EARLY, side));
    }
    auto late = [&]() -> int {
        if (!want_tail) return AECF_OK;
        AECF_TRY(launch_grad_gather(a, GATHER_LATE, side));
        const float* final_sums = a.sums;
        if (dp != nullptr) {
            AECF_TRY(launch_peer_sum(dev, dp, tail_layout(D, g.HSP).total, side));
            final_sums = static_cast<const float*>(dp->reduced[dp->rank]);
        }
        return launch_grad_finish(a, final_sums, side);
    };
    if (forked) AECF_CUDA_OK(cudaEventRecord(static_cast<cudaEvent_t>(gr->fork_event2), s));         // after the [dWv ; R] product
    if (gr->d_key) {                                         // dX = [dV | ds] . [Wv ; Qk]
        ScopedSite site(AECF_SITE_D_X);
        const aecf_gemm_desc d = gemm_desc(dev, dt, dt, dt, dt, AECF_K_MAJOR, AECF_MN_MAJOR, g.rows, D, KF, KF, D, D);
        AECF_TRY(aecf_gemm(&d, gr->d_kv, t->folded_w, nullptr, gr->d_key, w.gemm, w.gemm_bytes, s));
    }
    if (forked) {
        AECF_CUDA_OK(cudaStreamWaitEvent(side, static_cast<cudaEvent_t>(gr->fork_event2), 0));
        AECF_TRY(late());
        AECF_CUDA_OK(cudaEventRecord(static_cast<cudaEvent_t>(gr->join_event), side));
    }
    if (forked) AECF_CUDA_OK(cudaStreamWaitEvent(s, static_cast<cudaEvent_t>(gr->join_event), 0));
    else AECF_TRY(late());
    return AECF_OK;
}

}  // namespace aecf

using namespace aecf;

extern "C" {

size_t aecf_fusion_grad_sums_bytes(const aecf_pool_desc* desc) {
    Geometry g;
    if (geometry(desc, &g) != AECF_OK || !g.fold) return 0;
    return static_cast<size_t>(tail_layout(g.D, g.HSP).total) * sizeof(float);
}

size_t aecf_fusion_workspace_bytes(const aecf_pool_desc* desc) {
    Geometry g;
    if (geometry(desc, &g) != AECF_OK) return 0;
    Workspace w;
    carve(desc, g, nullptr, &w);
    return w.total;
}

int aecf_fusion_fwd(const aecf_pool_desc* desc, const aecf_fusion_tensors* t, void* workspace, size_t workspace_bytes,
                    void* stream) {
    Geometry g;
    AECF_TRY(geometry(desc, &g));
    if (!t || !t->query || !t->key || !t->in_proj_weight || !t->out_proj_weight || !t->q_proj || !t->kv || !t->ctx ||
        !t->out || !t->pooled || !workspace)
        return AECF_ERR_INVALID;
    if (g.B == 0) return AECF_OK;
    Workspace w;
    carve(desc, g, workspace, &w);
    if (workspace_bytes < w.total) return AECF_ERR_WORKSPACE;
    const int dt = g.dt, es = g.es, D = g.D, dev = desc->device;
    const bool bias = t->in_proj_bias != nullptr;
    const long long DD = static_cast<long long>(D) * D;

    if (!g.fold) {   // query projection (torch/nn/functional.py:5854); a shared query is projected once, in fp32
        ScopedSite site(AECF_SITE_Q_PROJ);
        const aecf_gemm_desc q = g.shared
            ? gemm_desc(dev, dt, dt, AECF_F32, dt, AECF_K_MAJOR, AECF_K_MAJOR, 1, D, D, D, D, D)
            : gemm_desc(dev, dt, dt, dt, dt, AECF_K_MAJOR, AECF_K_MAJOR, g.QR, D, D, D, D, D);
        AECF_TRY(aecf_gemm(&q, t->query, t->in_proj_weight, t->in_proj_bias, t->q_proj, w.gemm, w.gemm_bytes, stream));
    }
    if (g.fold) {
        // folded key projection: no K.  [Wv ; Qk] -> values + per-head scores in one pass over x -> pool -> out
        if (t->value || !t->scores || !t->folded_w) return AECF_ERR_INVALID;
        {   // q_proj = Wq q0 + bq and [Wv ; Qk] in one launch
            ScopedSite site(AECF_SITE_FOLD_PREPARE);
            AECF_TRY(aecf_fold_prepare_query(dev, dt, D, g.H, t->query, t->in_proj_weight, t->in_proj_bias,
                                             static_cast<float*>(t->q_proj), t->folded_w, stream));
        }
        {
            ScopedSite site(AECF_SITE_KV_PROJ);
            const aecf_gemm_desc v = gemm_desc(dev, dt, dt, dt, dt, AECF_K_MAJOR, AECF_K_MAJOR, g.rows, D, D, D, D, D);
            AECF_TRY(aecf_gemm_aux(&v, t->key, t->folded_w, bias ? at(t->in_proj_bias, 2 * D, es) : nullptr, t->kv, t->scores,
                                   g.H, g.HS, w.gemm, w.gemm_bytes, stream));
        }
        if (desc->row_index != nullptr)                          // unlisted samples: a zero context
            AECF_CUDA_OK(cudaMemsetAsync(t->ctx, 0, static_cast<size_t>(g.QR) * D * es, static_cast<cudaStream_t>(stream)));
        {
            ScopedSite site(AECF_SITE_POOL_FWD);
            AECF_TRY(aecf_pool_fwd_folded(desc, t->scores, t->kv, t->score_bias, t->ctx, t->pooled, t->entropy, t->mask_rate,
                                          t->masked, t->mask_bits, stream));
        }
    } else {
    {   // packed key/value projection (:5855); written straight into [rows, 2D] (no split copy, :5857-5863)
        ScopedSite site(AECF_SITE_KV_PROJ);
        if (!t->value) {
            const aecf_gemm_desc kv = gemm_desc(dev, dt, dt, dt, dt, AECF_K_MAJOR, AECF_K_MAJOR, g.rows, 2 * D, D, D, D, 2 * D);
            AECF_TRY(aecf_gemm(&kv, t->key, at(t->in_proj_weight, DD, es), bias ? at(t->in_proj_bias, D, es) : nullptr,
                               t->kv, w.gemm, w.gemm_bytes, stream));
        } else {
            const aecf_gemm_desc half = gemm_desc(dev, dt, dt, dt, dt, AECF_K_MAJOR, AECF_K_MAJOR, g.rows, D, D, D, D, 2 * D);
            AECF_TRY(aecf_gemm(&half, t->key, at(t->in_proj_weight, DD, es), bias ? at(t->in_proj_bias, D, es) : nullptr,
                               t->kv, w.gemm, w.gemm_bytes, stream));
            AECF_TRY(aecf_gemm(&half, t->value, at(t->in_proj_weight, 2 * DD, es),
                               bias ? at(t->in_proj_bias, 2 * D, es) : nullptr, at(t->kv, D, es), w.gemm, w.gemm_bytes, stream));
        }
    }
    if (desc->row_index != nullptr)
        AECF_CUDA_OK(cudaMemsetAsync(t->ctx, 0, static_cast<size_t>(g.QR) * D * es, static_cast<cudaStream_t>(stream)));
    {
        ScopedSite site(AECF_SITE_POOL_FWD);
        AECF_TRY(aecf_pool_fwd(desc, t->q_proj, t->kv, t->score_bias, t->ctx, t->pooled, t->entropy, t->mask_rate,
                               t->masked, t->mask_bits, stream));
    }
    }
    {   // out projection (:6653)
        ScopedSite site(AECF_SITE_OUT_PROJ);
        const aecf_gemm_desc o = gemm_desc(dev, dt, dt, dt, dt, AECF_K_MAJOR, AECF_K_MAJOR, g.QR, D, D, D, D, D);
        AECF_TRY(aecf_gemm(&o, t->ctx, t->out_proj_weight, t->out_proj_bias, t->out, w.gemm, w.gemm_bytes, stream));
    }
    return AECF_OK;
}

int aecf_fusion_bwd(const aecf_pool_desc* desc, const aecf_fusion_tensors* t, const aecf_fusion_grads* gr, void* workspace,
                    size_t workspace_bytes, void* stream) {
    Geometry g;
    AECF_TRY(geometry(desc, &g));
    if (!t || !gr || !workspace) return AECF_ERR_INVALID;
    if (!t->query || !t->key || !t->in_proj_weight || !t->out_proj_weight || !t->q_proj || !t->kv || !t->ctx ||
        !gr->d_out || !gr->d_ctx || !gr->d_kv)
        return AECF_ERR_INVALID;
    if (!g.shared && !gr->d_q_rows) return AECF_ERR_INVALID;
    if (g.B == 0) return AECF_OK;
    Workspace w;
    carve(desc, g, workspace, &w);
    if (workspace_bytes < w.total) return AECF_ERR_WORKSPACE;
    const int dt = g.dt, es = g.es, gdt = g.gdt, ges = g.ges, D = g.D, dev = desc->device;
    const long long DD = static_cast<long long>(D) * D;
    cudaStream_t s = static_cast<cudaStream_t>(stream);

    if (g.fold) {
        if (t->value || !t->scores || !t->folded_w) return AECF_ERR_INVALID;
        return folded_backward(desc, g, t, gr, w, s);
    }
    // ---- out-projection backward ----------------------------------------------------------------------
    if (gr->d_out_proj_bias) {
        ScopedSite site(AECF_SITE_D_OUT_BIAS);
        AECF_TRY(aecf_colsum(dev, dt, gdt, gr->d_out, g.QR, D, D, gr->d_out_proj_bias, w.colsum, w.colsum_bytes, stream));
    }
    if (gr->d_out_proj_weight) {                             // dWo = g^T ctx
        ScopedSite site(AECF_SITE_D_OUT_WEIGHT);
        const aecf_gemm_desc d = gemm_desc(dev, dt, dt, gdt, dt, AECF_MN_MAJOR, AECF_MN_MAJOR, D, D, g.QR, D, D, D);
        AECF_TRY(aecf_gemm(&d, gr->d_out, t->ctx, nullptr, gr->d_out_proj_weight, w.gemm, w.gemm_bytes, stream));
    }
    {                                                        // d_ctx = g Wo
        ScopedSite site(AECF_SITE_D_CTX);
        const aecf_gemm_desc d = gemm_desc(dev, dt, dt, dt, dt, AECF_K_MAJOR, AECF_MN_MAJOR, g.QR, D, D, D, D, D);
        AECF_TRY(aecf_gemm(&d, gr->d_out, t->out_proj_weight, nullptr, gr->d_ctx, w.gemm, w.gemm_bytes, stream));
    }
    if (desc->row_index != nullptr)
        AECF_CUDA_OK(cudaMemsetAsync(gr->d_kv, 0, static_cast<size_t>(g.rows) * 2 * D * es, s));
    {   // ---- fused recompute backward of the pool ---------------------------------------------------
        ScopedSite site(AECF_SITE_POOL_BWD);
        void* dq = g.shared ? static_cast<void*>(w.d_qp) : gr->d_q_rows;
        AECF_TRY(aecf_pool_bwd(desc, t->q_proj, t->kv, t->score_bias, gr->d_ctx, gr->d_pooled, gr->d_entropy, gr->d_kv, dq,
                               w.d_bias_kv, w.pool, w.pool_bytes, stream));
    }
    {   // ---- input gradients -----------------------------------------------------------------------------
        ScopedSite site(AECF_SITE_D_X);
        if (!t->value) {
            if (gr->d_key) {
                const aecf_gemm_desc d = gemm_desc(dev, dt, dt, dt, dt, AECF_K_MAJOR, AECF_MN_MAJOR, g.rows, D, 2 * D, 2 * D, D, D);
                AECF_TRY(aecf_gemm(&d, gr->d_kv, at(t->in_proj_weight, DD, es), nullptr, gr->d_key, w.gemm, w.gemm_bytes, stream));
            }
        } else {
            const aecf_gemm_desc d = gemm_desc(dev, dt, dt, dt, dt, AECF_K_MAJOR, AECF_MN_MAJOR, g.rows, D, D, 2 * D, D, D);
            if (gr->d_key)
                AECF_TRY(aecf_gemm(&d, gr->d_kv, at(t->in_proj_weight, DD, es), nullptr, gr->d_key, w.gemm, w.gemm_bytes, stream));
            if (gr->d_value)
                AECF_TRY(aecf_gemm(&d, at(gr->d_kv, D, es), at(t->in_proj_weight, 2 * DD, es), nullptr, gr->d_value, w.gemm,
                                   w.gemm_bytes, stream));
        }
    }
    if (gr->d_in_proj_weight) {   // ---- in-projection weight gradient (key / value rows) ----------------------
        {
            ScopedSite site(AECF_SITE_D_KV_WEIGHT);
            if (!t->value) {          // dW_kv = dKV^T X
                const aecf_gemm_desc d = gemm_desc(dev, dt, dt, gdt, dt, AECF_MN_MAJOR, AECF_MN_MAJOR, 2 * D, D, g.rows, 2 * D, D, D);
                AECF_TRY(aecf_gemm(&d, gr->d_kv, t->key, nullptr, at(gr->d_in_proj_weight, DD, ges), w.gemm, w.gemm_bytes, stream));
            } else {
                const aecf_gemm_desc d = gemm_desc(dev, dt, dt, gdt, dt, AECF_MN_MAJOR, AECF_MN_MAJOR, D, D, g.rows, 2 * D, D, D);
                AECF_TRY(aecf_gemm(&d, gr->d_kv, t->key, nullptr, at(gr->d_in_proj_weight, DD, ges), w.gemm, w.gemm_bytes, stream));
                AECF_TRY(aecf_gemm(&d, at(gr->d_kv, D, es), t->value, nullptr, at(gr->d_in_proj_weight, 2 * DD, ges), w.gemm,
                                   w.gemm_bytes, stream));
            }
        }
    }
    if (g.shared) {
        // ---- query side, shared query: dWq = d_qp (x) q0, d_query = d_qp . Wq, [d_bq | d_bk | d_bv] -- one launch
        if (gr->d_in_proj_weight || gr->d_query || gr->d_in_proj_bias) {
            ScopedSite site(AECF_SITE_D_QUERY);
            TimedLaunch timed(s);
            AECF_TRY(launch_query_tail(dt, gdt, D, w.d_qp, t->query, t->in_proj_weight, w.d_bias_kv, gr->d_in_proj_weight,
                                       gr->d_query, gr->d_in_proj_bias, s));
        }
        return AECF_OK;
    }
    if (gr->d_in_proj_weight) {   // ---- query rows of the in-projection weight gradient: dW_q = d_q^T Q -------------
        ScopedSite site(AECF_SITE_D_Q_WEIGHT);
        const aecf_gemm_desc d = gemm_desc(dev, dt, dt, gdt, dt, AECF_MN_MAJOR, AECF_MN_MAJOR, D, D, g.QR, D, D, D);
        AECF_TRY(aecf_gemm(&d, gr->d_q_rows, t->query, nullptr, gr->d_in_proj_weight, w.gemm, w.gemm_bytes, stream));
    }
    if (gr->d_query) {                // ---- gradient of the (unprojected) per-row queries ------------------------
        ScopedSite site(AECF_SITE_D_QUERY);
        const aecf_gemm_desc d = gemm_desc(dev, dt, dt, dt, dt, AECF_K_MAJOR, AECF_MN_MAJOR, g.QR, D, D, D, D, D);
        AECF_TRY(aecf_gemm(&d, gr->d_q_rows, t->in_proj_weight, nullptr, gr->d_query, w.gemm, w.gemm_bytes, stream));
    }
    if (gr->d_in_proj_bias) {         // ---- [d_bq | d_bk | d_bv] in the gradient dtype -------------------------
        ScopedSite site(AECF_SITE_D_IN_BIAS);
        AECF_TRY(aecf_colsum(dev, dt, AECF_F32, gr->d_q_rows, g.QR, D, D, w.d_bq, w.colsum, w.colsum_bytes, stream));
        TimedLaunch timed(s);
        const int n = 3 * D;
        if (gdt == AECF_BF16)
            AECF_CUDA_OK(launch_pdl(pack_in_bias_kernel<__nv_bfloat16>, dim3((n + 255) / 256), dim3(256), 0, s, w.d_bq, w.d_bias_kv,
                                    D, static_cast<__nv_bfloat16*>(gr->d_in_proj_bias)));
        else
            AECF_CUDA_OK(launch_pdl(pack_in_bias_kernel<float>, dim3((n + 255) / 256), dim3(256), 0, s, w.d_bq, w.d_bias_kv, D,
                                    static_cast<float*>(gr->d_in_proj_bias)));
        count_launch();
    }
    return AECF_OK;
}

}  // extern "C"
