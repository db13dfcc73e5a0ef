/*
 * aecf_b200 -- C ABI of the B200-native AECF fusion hot path.
 *
 * This is the drop-in boundary (SURVEY.md section 8b).  The reference has no FFI of its
 * own: its hot path is Python calling torch (reference aecf/AECFLayer.py:515-521 ->
 * torch.nn.MultiheadAttention, and :130-283 CurriculumMasking).  Each entry point below
 * replaces the stretch of that call chain cited next to it and is what a maintainer
 * would bind with ctypes (INTEGRATION.md shows the stub).
 *
 * Conventions
 *  - plain pointers and sizes only; every pointer is a DEVICE pointer unless marked host
 *  - the caller (torch) owns every buffer, including workspaces; nothing is allocated,
 *    freed or retained here; pointers are borrowed for the duration of the enqueue
 *  - every call is asynchronous on `stream` (a cudaStream_t passed as void*), never
 *    synchronises the host, and is re-entrant (autograd's worker thread calls the
 *    backward entry points)
 *  - return value: 0 or a negative aecf_status; nothing throws, exits or aborts
 *  - there is no CPU path: without a CUDA device every compute call returns
 *    AECF_ERR_CUDA
 *
 * Random stream contract (mirrored by oracle/philox.py, the CPU checker):
 *    Philox4x32-10, key = (seed & 0xffffffff, seed >> 32)
 *    counter = (row & 0xffffffff, row >> 32, offset & 0xffffffff,
 *               (stream << 28) | (head << 4) | block)
 *    row    = row0 + local row index (GLOBAL sample index: an N-rank batch-sharded run
 *             reproduces the 1-rank masks bit for bit)
 *    stream = 0 curriculum mask (head = 0), 1 attention dropout
 *    block  = m / 4 (< 16); lane m % 4 of the 4x32-bit output is the draw of token m
 *    u      = float(x) * 2^-32 + 2^-33   in (0, 1]
 *    mask keeps token m iff u <= keep_prob;  dropout keeps (head, m) iff u >= dropout_p
 */
#ifndef AECF_B200_H
#define AECF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(AECF_BUILDING_LIB)
#define AECF_API __attribute__((visibility("default")))
#else
#define AECF_API
#endif

#define AECF_ABI_VERSION 5
#define AECF_MAX_TOKENS 8

typedef enum aecf_status {
    AECF_OK = 0,
    AECF_ERR_INVALID = -1,      /* bad argument (null pointer, non-positive size, H does not divide D ...) */
    AECF_ERR_UNSUPPORTED = -2,  /* valid for the reference but outside what the kernels cover; no fallback */
    AECF_ERR_ALIGNMENT = -3,    /* a pointer or leading dimension is not 16-byte aligned */
    AECF_ERR_WORKSPACE = -4,    /* workspace too small */
    AECF_ERR_CUDA = -5          /* a CUDA runtime/driver call failed (see aecf_last_cuda_error) */
} aecf_status;

typedef enum aecf_dtype { AECF_F32 = 0, AECF_BF16 = 1 } aecf_dtype;

/* Operand layouts for aecf_gemm.  "K-major": the reduction index is contiguous. */
typedef enum aecf_layout { AECF_K_MAJOR = 0, AECF_MN_MAJOR = 1 } aecf_layout;

typedef enum aecf_gemm_impl { AECF_GEMM_AUTO = 0, AECF_GEMM_SIMT = 1, AECF_GEMM_TCGEN05 = 2 } aecf_gemm_impl;

/* ---- fused attention pool ------------------------------------------------------------
 * One descriptor for forward and backward.  All pool arithmetic is fp32; `dtype` is the
 * storage type of kv / ctx / d_ctx / d_kv (and of q, d_q when the query is per-row). */
typedef struct aecf_pool_desc {
    int32_t  device;          /* CUDA device ordinal the pointers live on */
    int32_t  dtype;           /* aecf_dtype */
    int64_t  batch;           /* B: rows in this call (>= 0; 0 is a no-op) */
    int32_t  num_tokens;      /* M: modality tokens per row, 1..AECF_MAX_TOKENS */
    int32_t  embed_dim;       /* D */
    int32_t  num_heads;       /* H, divides D; D/H must be a multiple of 16 bytes, at most 128 such chunks */
    int32_t  training;        /* attention module in training mode (enables dropout) */
    int32_t  masking;         /* 0: no CurriculumMasking stage; 1: module in training mode; 2: in eval mode */
    int32_t  min_active;      /* CurriculumMasking.min_active */
    int32_t  q_is_shared;     /* 1: one fp32 projected query [D] for all rows; 0: per-row [B, D] in dtype */
    float    base_mask_prob;  /* CurriculumMasking.base_mask_prob */
    float    entropy_target;  /* CurriculumMasking.entropy_target */
    float    dropout_p;       /* attention dropout (used only when training) */
    uint64_t seed;            /* Philox key */
    uint64_t offset;          /* Philox call offset, < 2^32 */
    uint64_t row0;            /* global index of local row 0 */
    int64_t  bias_stride_b;   /* score_bias strides in elements (0 broadcasts); token index is contiguous */
    int64_t  bias_stride_h;
    int64_t  kv_stride_b;     /* kv / d_kv strides in elements between rows and between tokens; 0, 0 means the */
    int64_t  kv_stride_m;     /* packed [B, M, 2D] layout (M*2D, 2D); a sequence-first [M, B, 2D] buffer is (2D, B*2D) */
    int32_t  fold_key;        /* whole-step entry points only: 1 = folded key projection (see "folded key projection") */
    int32_t  tgt_len;         /* S: fusion queries per sample; 0 or 1 = one (the hot path), see "several queries" below */
    /* CUDA-graph capture: a by-value (seed, offset) would be frozen into the graph.  When non-null, this DEVICE
     * pointer to {seed, offset} (two uint64) is read by the kernels at run time instead: key = seed, call offset =
     * low 32 bits of (offset + desc.offset); the caller advances the device-side offset between replays. */
    const uint64_t* rng_state;
    /* several queries per sample (tgt_len > 1) only */
    int64_t  q_stride_b;      /* ROW of query (b, s) in q / ctx / d_ctx / d_q and in the whole-step query / out / d_out: */
    int64_t  q_stride_s;      /*   b*q_stride_b + s*q_stride_s; (0, 0) = batch-first (S, 1); sequence-first is (1, B) */
    int64_t  bias_stride_s;   /* score_bias stride between the queries of a sample (0 broadcasts) */
    /* Fused CurriculumMasking.entropy_loss (reference aecf/AECFLayer.py:285-314; north_star: "the per-sample entropy_loss
     * term" in the fused kernel).  When loss_out is non-null, masking == 1 and one warp owns a sample (the streaming forward
     * kernel: embed_dim <= 64 sixteen-byte chunks), the forward also writes
     *     loss_out[0] = max(0, mean_b (nan_to_num(entropy[b], nan=0, posinf=1, neginf=0) - loss_target)^2)
     * Per-warp partial sums are folded per CTA and then by the last CTA to finish, each in index order: the result does not
     * depend on which CTA is last (no floating-point atomics).  Where the kernel in use does not carry the term, loss_out is
     * left untouched and aecf_pool_fwd_has_loss(desc) says so beforehand: the caller then runs aecf_entropy_loss_fwd. */
    float*   loss_out;        /* [1] fp32, nullable */
    void*    loss_workspace;  /* aecf_pool_loss_workspace_bytes() bytes, zeroed ONCE by the caller (the kernel re-arms it) */
    float    loss_target;     /* entropy_target * log(_last_seq_len), the value CurriculumMasking.entropy_loss would use */
    /* Whole-step entry points only: 1 = mixed precision (see "mixed precision" there): the parameter pointers of
     * aecf_fusion_tensors are bf16 shadows of fp32 parameters and the parameter gradients of aecf_fusion_grads are fp32.
     * Needs dtype == AECF_BF16; 0 = every tensor not marked fp32 is in dtype; any other value is AECF_ERR_INVALID. */
    int32_t  param_grads_f32;
    /* Row indirection (reference xrays/train_xrays_example.py:202-222 gathers the rows where both modalities are present,
     * pools them and scatters the result back; here the pool kernels do both ends themselves).  With row_index non-null,
     * `batch` counts the LISTED rows: row i of this call -- its Philox row (row0 + i), its pooled / entropy / mask_rate /
     * masked / mask_bits outputs, its d_pooled / d_entropy -- is sample row_index[i] of kv / scores / ctx / d_ctx / d_kv, which
     * keep their full-batch layout of `src_rows` samples.  ctx rows of unlisted samples are zeroed by the whole-step forward,
     * their d_kv rows by the whole-step backward, so the products around the pool simply run over all src_rows samples.
     * Needs a shared query (q_is_shared), one query per sample, no score_bias. */
    const int64_t* row_index; /* [batch] DEVICE, distinct values in [0, src_rows); null: the identity */
    int64_t  src_rows;        /* samples in the buffers when row_index is set */
} aecf_pool_desc;

/* Several queries per sample (tgt_len = S > 1; reference aecf/AECFLayer.py:415 takes any [B, S, D] query).  Every
 * (b, s) pair is a row of its own for the softmax, the dropout draws, the head mean and the CurriculumMasking
 * stage; the S rows of a sample share its M keys and values, whose gradients sum over them.  In this mode
 *   - the query is per row (q_is_shared = 0) and the key projection is not folded (fold_key = 0);
 *   - q / ctx / d_ctx / d_q hold B*S rows of D at b*q_stride_b + s*q_stride_s;
 *   - pooled / masked are [B, S, M], entropy / mask_rate / mask_bits / d_entropy [B, S], d_pooled [B, S, M], all
 *     b-major whatever the query layout (torch returns the weights as [B, S, M], functional.py:6657);
 *   - the Philox row of (b, s) is (row0 + b) * S + s, so S == 1 is the contract above unchanged;
 *   - score_bias element (b, h, s, m) sits at b*bias_stride_b + h*bias_stride_h + s*bias_stride_s + m.
 * kv / d_kv keep their [B, M, 2D] layout and strides. */

/* Forward: scale, per-head scores, softmax, dropout, weighted value sum, head mean, and the whole
 * CurriculumMasking stage.  Replaces torch/nn/functional.py:6632-6647, 6657-6659 and reference
 * aecf/AECFLayer.py:130-283 (~45 ATen launches, >= 5 host syncs) with one launch.
 *   q          [D] fp32 (q_is_shared) or [B, D] dtype : projected query, NOT yet scaled
 *   kv         [B, M, 2D] dtype : projected keys (cols 0..D) and values (cols D..2D); other row/token
 *              strides via kv_stride_b / kv_stride_m (d_kv of the backward uses the same strides)
 *   score_bias nullable fp32, additive (key_padding_mask / attn_mask as torch merges them,
 *              functional.py:6608-6620); element (b, h, m) at b*bias_stride_b + h*bias_stride_h + m
 *   ctx        [B, D] dtype          out: per-head weighted value sum, heads concatenated
 *   pooled     [B, M] fp32           out: info['attention_weights'] (head mean, post-dropout)
 *   entropy    [B] fp32, nullable    out: info['entropy']
 *   mask_rate  [B] fp32, nullable    out: info['mask_rate']
 *   masked     [B, M] fp32, nullable out: info['masked_attention_weights']
 *   mask_bits  [B] u8, nullable      out: bit m set iff token m is active after min_active repair */
AECF_API int aecf_pool_fwd(const aecf_pool_desc* desc, const void* q, const void* kv, const float* score_bias,
                  void* ctx, float* pooled, float* entropy, float* mask_rate, float* masked,
                  uint8_t* mask_bits, void* stream);
AECF_API size_t aecf_pool_loss_workspace_bytes(void);
/* 1 when aecf_pool_fwd / aecf_pool_fwd_folded (`folded` != 0) / aecf_fusion_fwd with this descriptor write desc->loss_out */
AECF_API int aecf_pool_fwd_has_loss(const aecf_pool_desc* desc, int32_t folded);

/* Backward: recomputes the attention weights from q/kv (nothing from forward is stored; this is what
 * use_checkpoint= asked for, reference aecf/AECFLayer.py:501-512) and produces every activation
 * gradient of the pool in one launch plus a tiny deterministic finalize.
 *   d_ctx      [B, D] dtype
 *   d_pooled   [B, M] fp32, nullable : gradient w.r.t. info['attention_weights']
 *   d_entropy  [B] fp32, nullable    : gradient w.r.t. info['entropy'] (eval mode only, :151-156)
 *   d_kv       [B, M, 2D] dtype      out
 *   d_q        q_is_shared ? [D] fp32 (summed over rows) : [B, D] dtype   out
 *   d_bias_kv  [2D] fp32, nullable   out: column sums of d_kv (gradient of in_proj_bias[D:])
 *   workspace  >= aecf_pool_bwd_workspace_bytes(desc) bytes */
AECF_API int aecf_pool_bwd(const aecf_pool_desc* desc, const void* q, const void* kv, const float* score_bias,
                  const void* d_ctx, const float* d_pooled, const float* d_entropy,
                  void* d_kv, void* d_q, float* d_bias_kv,
                  void* workspace, size_t workspace_bytes, void* stream);
AECF_API size_t aecf_pool_bwd_workspace_bytes(const aecf_pool_desc* desc);

/* ---- folded key projection (one query shared by all rows) ------------------------------------
 * With a single fusion query the keys never need to exist:
 *     score[b, h, m] = scale * q_h . (Wk_h x[b, m] + bk_h) = x[b, m] . Qk[h] + const(h),
 *     Qk[h] = scale * Wk_h^T q_h  (one D-vector per head),
 * and const(h) shifts all tokens of a head alike, so it drops out of the softmax.  The value projection GEMM
 * produces the scores as a side output in the same pass over x (aecf_gemm_aux, B = [Wv ; Qk]); the pool kernels
 * then read the values and the scores only.  Backward: dK = ds (x) (scale q) has rank H per row, so instead of
 * dK the kernel stores ds itself next to dV, d_vs[row] = [dV (D) | ds (HSP)], and the two GEMMs that follow
 * contract over D + HSP:  dX = d_vs . [Wv ; Qk]   and   [dWv ; R] = d_vs^T . X,  R[h] = sum_{b,m} ds[b,h,m] x[b,m],
 * from which dWk[h*hd + j] = scale * q[h*hd + j] * R[h] and d q[h*hd + j] = scale * Wk[h*hd + j] . R[h].
 * Half the projection FLOPs and 45 % of the pool kernels' HBM bytes disappear; the arithmetic is re-associated,
 * so results differ from the unfolded path by rounding only (fp32: ~1e-6 relative).
 * These entry points take matrices of B*M rows; kv_stride_b / kv_stride_m of the descriptor are in ROWS here
 * ((0, 0) = (M, 1): row b*M + m; a sequence-first batch is (1, B)).
 *   scores [B*M, HS]  fp32, HS = num_heads rounded up to 4
 *   v      [B*M, D]   dtype
 *   d_vs   [B*M, D + HSP] dtype, HSP = aecf_fold_score_cols(dtype, num_heads) (16-byte multiple)
 *   q_proj [D] fp32   (only its product with sum ds enters d_bias_kv[0 .. D), analytically zero)
 * d_bias_kv as in aecf_pool_bwd. */
AECF_API int aecf_fold_score_cols(int32_t dtype, int32_t num_heads);
AECF_API int aecf_pool_fwd_folded(const aecf_pool_desc* desc, const float* scores, const void* v, const float* score_bias,
                         void* ctx, float* pooled, float* entropy, float* mask_rate, float* masked,
                         uint8_t* mask_bits, void* stream);
AECF_API int aecf_pool_bwd_folded(const aecf_pool_desc* desc, const void* q_proj, const float* scores, const void* v,
                         const float* score_bias, const void* d_ctx, const float* d_pooled, const float* d_entropy,
                         void* d_vs, float* d_bias_kv, void* workspace, size_t workspace_bytes, void* stream);
/* Forward preparation: folded_w [D + HSP, D] dtype = [ Wv ; Qk (H rows) ; zero rows ] from the projected query
 * q_proj [D] fp32 and in_proj_weight [3D, D]. */
AECF_API int aecf_fold_prepare(int32_t device, int32_t dtype, int32_t embed_dim, int32_t num_heads, const float* q_proj,
                      const void* in_proj_weight, void* folded_w, void* stream);
/* The same from the UNPROJECTED shared query [D] (dtype): also computes and writes q_proj [D] fp32 = Wq query + bq
 * (torch/nn/functional.py:5854; in_proj_bias nullable) -- one launch in front of the forward GEMM instead of two. */
AECF_API int aecf_fold_prepare_query(int32_t device, int32_t dtype, int32_t embed_dim, int32_t num_heads, const void* query,
                            const void* in_proj_weight, const void* in_proj_bias, float* q_proj, void* folded_w,
                            void* stream);
/* Backward completion: from g = [dWv ; R] ([D + HSP, D] fp32, the output of the d_vs^T . X product) write
 * d_in_proj_weight rows [D, 2D) (dWk) and [2D, 3D) (dWv) in dtype (either may be skipped with a null
 * d_in_proj_weight) and d_q_proj [D] fp32 (+= nothing: overwritten). */
AECF_API int aecf_fold_finish(int32_t device, int32_t dtype, int32_t embed_dim, int32_t num_heads, const float* g,
                     const float* q_proj, const void* in_proj_weight, void* d_in_proj_weight, float* d_q_proj,
                     void* stream);

/* ---- projections ------------------------------------------------------------------------
 * C[m, n] = sum_k A[m, k] * B[n, k] (+ bias[n]) (+ C if accumulate), fp32 accumulation.
 * Replaces torch.nn.functional.linear at torch/nn/functional.py:5854-5855, 6653 and the four
 * matmuls autograd derives from them.
 *   a_layout K_MAJOR : A(i, k) at A[i*lda + k]     MN_MAJOR : A(i, k) at A[k*lda + i]
 *   b_layout K_MAJOR : B(j, k) at B[j*ldb + k]     MN_MAJOR : B(j, k) at B[k*ldb + j]
 *   C(i, j) at C[i*ldc + j]; bias has dtype_bias and n elements
 * impl TCGEN05 needs bf16 A and B; AUTO picks it whenever it applies. */
typedef struct aecf_gemm_desc {
    int32_t device;
    int32_t dtype_a, dtype_b, dtype_c, dtype_bias;   /* aecf_dtype */
    int32_t a_layout, b_layout;                      /* aecf_layout */
    int32_t accumulate;                              /* 1: C += ... */
    int32_t impl;                                    /* aecf_gemm_impl */
    int64_t m, n, k;
    int64_t lda, ldb, ldc;
} aecf_gemm_desc;

AECF_API int aecf_gemm(const aecf_gemm_desc* desc, const void* A, const void* B, const void* bias, void* C,
              void* workspace, size_t workspace_bytes, void* stream);
AECF_API size_t aecf_gemm_workspace_bytes(const aecf_gemm_desc* desc);

/* Same product with a narrow fp32 side output taken from extra rows of B (the folded key projection
 * computes the attention scores this way, in the same pass over A as the value projection):
 *   C[i, j]   = sum_k A[i, k] * B[j, k] + bias[j]           j < n            (dtype_c, ldc)
 *   aux[i, j] = sum_k A[i, k] * B[n + j, k]                 j < aux_cols     (fp32, aux_ld)
 * B has n + aux_rows rows, aux_rows = aux_cols rounded up to 16 bytes of dtype_b; aux_ld >= aux_cols rounded
 * up to 4 and the columns aux_cols .. of each aux row up to that multiple are written too (with the products
 * of the padding rows of B).  aux_cols <= 32.  On the tcgen05 path (bf16, n % 32 == 0, B K-major) it is ONE
 * launch: 128 x 192 tiles, the side columns leave the epilogue as fp32 straight from the accumulator. */
AECF_API int aecf_gemm_aux(const aecf_gemm_desc* desc, const void* A, const void* B, const void* bias, void* C,
                           float* aux, int32_t aux_cols, int64_t aux_ld, void* workspace, size_t workspace_bytes,
                           void* stream);

/* ---- small reductions ------------------------------------------------------------------
 * out[c] = sum_r x[r*ld + c] for a [rows, cols] matrix, fp32 accumulation, deterministic.
 * (gradient of out_proj.bias; torch/nn/functional.py:6653 backward).  workspace >= the _bytes query. */
AECF_API int aecf_colsum(int32_t device, int32_t dtype_x, int32_t dtype_out, const void* x, int64_t rows,
                int64_t cols, int64_t ld, void* out, void* workspace, size_t workspace_bytes, void* stream);
AECF_API size_t aecf_colsum_workspace_bytes(int64_t rows, int64_t cols);

/* CurriculumMasking.entropy_loss (reference aecf/AECFLayer.py:285-314):
 * loss[0] = max(0, mean((nan_to_num(e) - target)^2)), deterministic single-block reduction. */
AECF_API int aecf_entropy_loss_fwd(int32_t device, const float* entropy, int64_t n, float target, float* loss,
                          void* stream);
/* d_entropy[i] = d_loss[0] * 2 * (e[i] - target) / n   (zero where e[i] is not finite) */
AECF_API int aecf_entropy_loss_bwd(int32_t device, const float* entropy, int64_t n, float target,
                          const float* d_loss, float* d_entropy, void* stream);

/* Standalone CurriculumMasking.forward / compute_entropy on caller-supplied weights [rows, len] fp32,
 * len <= 64 (reference aecf/AECFLayer.py:101-283; the pool kernel carries the same stage fused).
 *   mode 1: training (mask, repair, renormalise)   2: eval (weights unchanged, entropy of the input)
 *        3: entropy only (compute_entropy).  masked / entropy / mask_rate are nullable. */
AECF_API int aecf_curriculum_mask(int32_t device, const float* weights, int64_t rows, int32_t len, int32_t mode,
                                  float base_mask_prob, int32_t min_active, uint64_t seed, uint64_t offset,
                                  uint64_t row0, float* masked, float* entropy, float* mask_rate, void* stream);
/* Backward of the mode-1 call: d_weights [rows, len] for d_masked [rows, len].  The mask is REDRAWN from the same
 * (seed, offset, row0); mask, top-k repair set and entropy carry no gradient, the renormalisations do (the reference's
 * final_weights = weights * mask / sum keeps its graph, aecf/AECFLayer.py:262-272). */
AECF_API int aecf_curriculum_mask_bwd(int32_t device, const float* weights, int64_t rows, int32_t len, float base_mask_prob,
                                      int32_t min_active, uint64_t seed, uint64_t offset, uint64_t row0,
                                      const float* d_masked, float* d_weights, void* stream);
/* d_weights = d_entropy * d clamp(-sum xlogy(w, w), 0, log len) / d w */
AECF_API int aecf_entropy_bwd(int32_t device, const float* weights, int64_t rows, int32_t len,
                              const float* d_entropy, float* d_weights, void* stream);

/* Projection-free single-head attention of the functional fast path
 * (reference aecf/AECFLayer.py:556-581): out[b, s, :] = softmax_t(q[b,s]·k[b,t] / sqrt(D)) · v[b,t]. */
AECF_API int aecf_sdpa_fwd(int32_t device, int32_t dtype, const void* q, const void* k, const void* v, void* out,
                  int64_t batch, int32_t tgt_len, int32_t src_len, int32_t embed_dim, void* stream);
/* Its backward (the reference's function is plain differentiable torch): d_q [B, tgt, D], d_k / d_v [B, src, D] for
 * d_out [B, tgt, D]; nothing is stored by the forward, the weights are recomputed.  workspace >= 2 * B * tgt_len floats. */
AECF_API int aecf_sdpa_bwd(int32_t device, int32_t dtype, const void* q, const void* k, const void* v, const void* d_out,
                  void* d_q, void* d_k, void* d_v, void* workspace, size_t workspace_bytes, int64_t batch,
                  int32_t tgt_len, int32_t src_len, int32_t embed_dim, void* stream);

/* ---- parameter shadow (mixed precision) ---------------------------------------------------------
 * One launch rounds up to AECF_PARAM_CAST_MAX_SEGMENTS fp32 segments to bf16 (round to nearest even, like
 * Tensor.bfloat16(); NaN stays NaN, +-inf stays +-inf, values past the bf16 range round to +-inf) into one block:
 * segment i of counts[i] elements lands at element offset(i) of dst, offset(0) = 0 and
 * offset(i + 1) = offset(i) + counts[i] rounded up to 8, so every segment starts on a 16-byte boundary (a valid
 * GEMM / TMA operand).  Padding elements are not written.  src / counts are HOST arrays of `segments` entries
 * (device pointers / element counts); dst must be 16-byte aligned. */
#define AECF_PARAM_CAST_MAX_SEGMENTS 8
AECF_API int aecf_param_cast(int32_t device, int32_t segments, const float* const* src, const int64_t* counts, void* dst,
                             void* stream);

/* ---- whole-step entry points -------------------------------------------------------------
 * The complete forward and backward of MultimodalAttentionPool (reference aecf/AECFLayer.py:515-541 and
 * the autograd graph behind it) as one call each, so the host pays one FFI crossing per direction instead
 * of one per kernel.  They run exactly the calls above, in order, on `stream`.
 * All pointers are device pointers; nullable ones are marked.  `dtype` of the descriptor is the type of
 * every tensor not marked fp32.
 *
 * Mixed precision (desc->param_grads_f32 = 1, dtype = AECF_BF16): fp32 master parameters, bf16 compute, as
 * torch.autocast trains.  The caller rounds the fp32 parameters to bf16 once per forward (aecf_param_cast) and passes
 * those shadows as in_proj_weight / in_proj_bias / out_proj_weight / out_proj_bias (and, with a shared query, as
 * query); the forward and the backward then compute exactly what dtype = AECF_BF16 computes with those parameters.
 * The parameter gradients -- d_in_proj_weight, d_in_proj_bias, d_out_proj_weight, d_out_proj_bias and, with a shared
 * query, d_query -- are written in fp32, from the fp32 values the bf16 call would have rounded: rounded to bf16
 * they are bit for bit the bf16 call's gradients.  Every other tensor (key, value, per-row query and their
 * gradients, out, ctx, d_out ...) stays bf16. */
typedef struct aecf_fusion_tensors {
    /* inputs */
    const void*  query;            /* q_is_shared ? [D] : [B, D] */
    const void*  key;              /* [B*M, D]; rows ordered like kv (b-major, or m-major when kv_stride_* say so) */
    const void*  value;            /* nullable: separate value tensor, same layout as key */
    const void*  in_proj_weight;   /* [3D, D] */
    const void*  in_proj_bias;     /* [3D], nullable */
    const void*  out_proj_weight;  /* [D, D] */
    const void*  out_proj_bias;    /* [D], nullable */
    const float* score_bias;       /* nullable, see aecf_pool_fwd */
    /* forward results that the backward reads again (the caller keeps them alive) */
    void*  q_proj;                 /* q_is_shared ? [D] fp32 : [B, D] */
    void*  kv;                     /* [B*M, 2D]; folded key projection: [B*M, D] (the values only) */
    void*  ctx;                    /* [B, D] */
    /* forward outputs */
    void*    out;                  /* [B, D] */
    float*   pooled;               /* [B, M] fp32 */
    float*   entropy;              /* [B] fp32, nullable */
    float*   mask_rate;            /* [B] fp32, nullable */
    float*   masked;               /* [B, M] fp32, nullable */
    uint8_t* mask_bits;            /* [B], nullable */
    /* folded key projection (desc->fold_key): forward results the backward reads again; kv is then [B*M, D]
     * (values only) and d_kv of aecf_fusion_grads [B*M, D + HSP] */
    float*   scores;               /* [B*M, HS] fp32 */
    void*    folded_w;             /* [D + HSP, D] */
} aecf_fusion_tensors;

/* Cross-rank sum of the parameter gradients INSIDE the backward (csrc/grad_tail.cu; north_star item 3).  Every rank maps
 * every rank's buffers (CUDA IPC, aecf_b200.dp.GradientSync) and must have peer access enabled.  The raw gradient sums of
 * the folded backward -- [dWv ; R], dWo, colsum(d_out), the pool kernel's bias sums: aecf_fusion_grad_sums_bytes(desc)
 * bytes of fp32, about half the parameter count because dWk, dWq and d_query are linear images of R -- are summed over the
 * ranks IN FP32 by one kernel (flag barrier; rank r sums slice r of all ranks' buffers in rank order and stores it into
 * every rank's `reduced` buffer; flag barrier), and only then converted to the parameter dtype, so an N-rank run rounds once,
 * like a 1-rank run.  The kernel runs on the side stream next to the dX product.  Host arrays of `world` DEVICE pointers. */
typedef struct aecf_dp_desc {
    int32_t world, rank;      /* world <= 8 (one NVLink node) */
    int32_t average;          /* 1: divide the sums by world */
    int32_t reserved0;
    void* const* sums;        /* [world] every rank's raw-sum buffer as mapped in THIS process (this rank's is written here) */
    void* const* reduced;     /* [world] every rank's reduced-sum buffer */
    void* const* flags;       /* [world] every rank's flag block, aecf_peer_flag_bytes() bytes, zeroed once */
} aecf_dp_desc;

typedef struct aecf_fusion_grads {
    const void*  d_out;            /* [B, D] */
    const float* d_pooled;         /* [B, M] fp32, nullable */
    const float* d_entropy;        /* [B] fp32, nullable (eval mode) */
    /* scratch the caller provides */
    void* d_ctx;                   /* [B, D] */
    void* d_kv;                    /* [B*M, 2D]; folded key projection: [B*M, D + HSP] (= [dV | ds]) */
    void* d_q_rows;                /* [B, D]; only when !q_is_shared */
    /* results; a null pointer skips that gradient */
    void* d_key;                   /* [B*M, D] */
    void* d_value;                 /* [B*M, D], only with a separate value */
    void* d_query;                 /* q_is_shared ? [D] : [B, D] */
    void* d_in_proj_weight;        /* [3D, D] */
    void* d_in_proj_bias;          /* [3D] */
    void* d_out_proj_weight;       /* [D, D] */
    void* d_out_proj_bias;         /* [D] */
    /* Folded backward: the small kernels that finish the parameter gradients (split-K folds, column
     * sums, the rank-H key/query terms, conversion to dtype; csrc/grad_tail.cu) run on `side_stream` NEXT TO the products on
     * `stream`: fork_event is recorded on `stream` after the pool backward (the column sums of d_out and the dWo fold then run
     * next to the [dWv ; R] product), fork_event2 after that product (the rest runs next to dX), join_event on `side_stream` after the last of them, and
     * `stream` waits for it before the call returns.  Any of the four null: everything on `stream`, in order.
     * The caller owns stream and events (cudaStream_t / cudaEvent_t handles); capture into a CUDA graph works as usual. */
    void* side_stream;
    void* fork_event;
    void* fork_event2;
    void* join_event;
    const aecf_dp_desc* dp;        /* nullable: sum the gradients over the ranks inside the backward (see aecf_dp_desc) */
} aecf_fusion_grads;

AECF_API int aecf_fusion_fwd(const aecf_pool_desc* desc, const aecf_fusion_tensors* t, void* workspace,
                             size_t workspace_bytes, void* stream);
AECF_API int aecf_fusion_bwd(const aecf_pool_desc* desc, const aecf_fusion_tensors* t, const aecf_fusion_grads* g,
                             void* workspace, size_t workspace_bytes, void* stream);
AECF_API size_t aecf_fusion_workspace_bytes(const aecf_pool_desc* desc);
/* bytes of ONE raw-sum (or reduced-sum) buffer of aecf_dp_desc for this descriptor; 0 where the backward has no fused tail
 * (unfolded key projection, per-row queries) */
AECF_API size_t aecf_fusion_grad_sums_bytes(const aecf_pool_desc* desc);

/* ---- data-parallel all-reduce over NVLink peer memory ------------------------------------------------
 * In-place sum (or mean) of one gradient bucket across the W <= 8 ranks of a node, one kernel per rank over peer
 * mappings of every rank's bucket (csrc/peer_allreduce.cu: barrier, each rank reduces its slice from all buckets in
 * rank order and stores it into all buckets, barrier).  Results are bit-identical on every rank.  The reference has no
 * distributed code; this replaces the NCCL all-reduce a data-parallel training loop would issue after the backward.
 *   peer_data[r]  : HOST array of W DEVICE pointers -- rank r's bucket as mapped in this process (CUDA IPC); all
 *                   buckets hold `count` elements padded to a multiple of 16 bytes
 *   peer_flags[r] : HOST array of W DEVICE pointers -- rank r's flag block, aecf_peer_flag_bytes() bytes, zeroed once
 * The caller maps the buffers (aecf_peer_export / aecf_peer_import below; aecf_b200.dp does it that way) and must have enabled peer
 * access (aecf_peer_enable_access).  Every rank must make the same sequence of calls.  Graph-capturable: the call
 * epoch lives in the flag block and is advanced by the kernel. */
typedef struct aecf_peer_desc {
    int32_t device, dtype, world, rank;
    int64_t count;
    int32_t average;          /* 1: divide the sum by world */
    int32_t grid_limit;       /* 0 = default (32 CTAs) */
} aecf_peer_desc;
AECF_API size_t aecf_peer_flag_bytes(void);
AECF_API int    aecf_peer_enable_access(int32_t device, int32_t peer_device);
AECF_API int    aecf_peer_allreduce(const aecf_peer_desc* desc, void* const* peer_data, void* const* peer_flags, void* stream);
/* CUDA IPC for those buffers.  export: the 64-byte IPC handle of the allocation `ptr` lies in and ptr's offset inside it
 * (the bytes travel to the other ranks by any means).  import: opens a handle in the context of `device` -- THIS rank's GPU,
 * so that its kernels can address the memory -- and returns the allocation's base; the buffer is at base + offset.  A
 * handle must be imported once per process (keep a cache keyed by its bytes); mappings live until the process exits. */
AECF_API int    aecf_peer_export(int32_t device, const void* ptr, void* handle64, int64_t* offset);
AECF_API int    aecf_peer_import(int32_t device, const void* handle64, void** base_out);

/* ---- per-kernel timing (CUDA events recorded next to each launch, on the launching stream) ------------- */
typedef enum aecf_site {
    AECF_SITE_OTHER = 0, AECF_SITE_Q_PROJ, AECF_SITE_KV_PROJ, AECF_SITE_POOL_FWD, AECF_SITE_OUT_PROJ,
    AECF_SITE_D_OUT_BIAS, AECF_SITE_D_OUT_WEIGHT, AECF_SITE_D_CTX, AECF_SITE_POOL_BWD, AECF_SITE_POOL_BWD_FINALIZE,
    AECF_SITE_D_X, AECF_SITE_D_KV_WEIGHT, AECF_SITE_D_Q_WEIGHT, AECF_SITE_D_QUERY, AECF_SITE_D_IN_BIAS,
    AECF_SITE_ENTROPY_LOSS, AECF_SITE_FOLD_PREPARE, AECF_SITE_FOLD_FINISH, AECF_SITE_GRAD_GATHER, AECF_SITE_GRAD_PEER_SUM,
    AECF_SITE_GRAD_FINISH, AECF_SITE_PARAM_CAST, AECF_SITE_COUNT
} aecf_site;
AECF_API int         aecf_timing_enable(int32_t enable);                    /* clears earlier records */
AECF_API int         aecf_timing_collect(float* total_ms, int32_t* launches); /* arrays of AECF_SITE_COUNT; syncs */
AECF_API const char* aecf_timing_site_name(int32_t site);
AECF_API const char* aecf_timing_site_gemm_kernel(int32_t site);            /* which GEMM kernel that site launched last ("" if none) */

/* ---- diagnostics ----------------------------------------------------------------------- */
AECF_API int         aecf_abi_version(void);
AECF_API const char* aecf_strerror(int status);
AECF_API const char* aecf_last_cuda_error(void);      /* host string, thread-local */
AECF_API uint64_t    aecf_launch_count(void);         /* kernels launched by this library since load */
AECF_API const char* aecf_build_info(void);           /* "sm_100a nvcc 12.9 ..." */
AECF_API const char* aecf_gemm_last_kernel(void);     /* host string, thread-local: which kernel the last aecf_gemm[_aux] call of this
                                                         thread launched, e.g. "tcgen05 1sm bn192 cluster2 epi1", "tcgen05 2sm bn256 ew4", "simt" */
AECF_API const char* aecf_pool_last_kernel(void);     /* host string, thread-local: which pool kernel and schedule the last pool launch
                                                         of this thread took, e.g. "stream M=3 J=1 PAD=0 fold=1 warps=24 rows_per_warp=19
                                                         ctas=148", "slice ... grid=N", "bwd grid-stride ... grid=G passes=P",
                                                         "bwd chunked ... grid=G chunk=C", "multi fwd ... grid=N", "multi bwd ... passes=P" */

#ifdef __cplusplus
}
#endif
#endif /* AECF_B200_H */
