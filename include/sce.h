/* sce.h — C ABI of the B200-native ensemble sparse-autoencoder training engine (libsce.so).
 *
 * The reference (HoagyC/sparse_coding @ 69c5ae0) has no FFI layer: its boundary for this path is the Python
 * protocol DictSignature / FunctionalEnsemble (autoencoders/ensemble.py:15-22, 68-193). This library sits
 * UNDERNEATH that protocol: sparse_coding_b200.FunctionalEnsemble keeps the reference's Python surface and
 * forwards the arithmetic of `step_batch` to the entry points below through ctypes (see INTEGRATION.md for the
 * binding a maintainer of the reference would add).
 *
 * Conventions: plain pointers and sizes only (no torch types); device pointers are borrowed — the caller (torch)
 * owns parameters, optimiser moments and the workspace, which are updated IN PLACE exactly as
 * FunctionalEnsemble.step_batch does (ensemble.py:182-191); no device allocation and no C++ exception crosses
 * the ABI; every call returns 0 on success or a negative sce_status, with a thread-local message available from
 * sce_last_error(); work is enqueued asynchronously on the caller's CUDA stream (`stream` is a cudaStream_t
 * passed as void*); calls on different plans are re-entrant, calls on the same plan are not thread-safe.
 */
#ifndef SCE_H_
#define SCE_H_

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SCE_VERSION 201 /* major*10000 + minor*100 + patch */

typedef enum sce_status {
  SCE_OK = 0,
  SCE_ERR_INVALID = -1,    /* bad argument / unsupported shape */
  SCE_ERR_CUDA = -2,       /* a CUDA runtime or driver call failed */
  SCE_ERR_WORKSPACE = -3,  /* workspace too small / misaligned */
  SCE_ERR_NO_DEVICE = -4   /* no sm_100 device / driver entry point missing */
} sce_status;

/* Which reference signature the plan reproduces. */
typedef enum sce_variant {
  SCE_TIED = 0,   /* FunctionalTiedSAE.loss   (sae_ensemble.py:135-162); + coef_mask = FunctionalMaskedTiedSAE (:347-373) */
  SCE_UNTIED = 1, /* FunctionalSAE.loss       (sae_ensemble.py:53-78);   + coef_mask = FunctionalMaskedSAE     (:418-444) */
  SCE_TOPK = 2    /* TopKEncoder.loss         (topk_encoder.py:29-40) */
} sce_variant;

/* How the Adam step counter behaves (SURVEY.md Q2). */
typedef enum sce_adam_count {
  SCE_ADAM_FROZEN_T1 = 0, /* the reference: step_batch drops torchopt's incremented count (ensemble.py:185-189) */
  SCE_ADAM_STANDARD = 1   /* bias correction with the true step number */
} sce_adam_count;

/* How an fp32 GEMM operand is carried to the tensor cores (DESIGN.md section 2). Both reach the reference's fp32
 * results within the 1e-4 bar; they differ in cost and in the range of values they can hold.
 *   BF16X3: x = hi + lo, two bf16 planes; product = hi*hi + hi*lo + lo*hi, three kind::f16 passes. fp32 range.
 *   F16F8 : x = h + l, h = fp16(x); the dominant h*h runs as one kind::f16 pass, the two cross terms (which need
 *           ~3 significant bits) as kind::f8f6f4 E5M2 passes at twice the rate: 2 pass-equivalents instead of 3.
 *           Operand values must fit fp16 (|v| < 65504; magnitudes below ~1e-4 lose relative precision) — true for
 *           language-model activations, which the reference itself stores as fp16 (activation_dataset.py:294-299, 364, 404-412).
 *           Needs d % 16 == 0 and n % 16 == 0.
 *   AUTO  : F16F8 when the shape allows it, else BF16X3 (env SCE_ARITH=bf16x3|f16f8 overrides AUTO). */
typedef enum sce_arith { SCE_ARITH_AUTO = 0, SCE_ARITH_BF16X3 = 1, SCE_ARITH_F16F8 = 2 } sce_arith;

/* Static description of one stacked ensemble (FunctionalEnsemble.__init__, ensemble.py:69-97). */
typedef struct sce_desc {
  int variant;          /* sce_variant */
  int n_models;         /* M: models stacked on dim 0 */
  int d;                /* activation width, multiple of 8 */
  int n;                /* dictionary rows (stack size for masked variants), multiple of 8 */
  int batch_max;        /* largest batch this plan will see (the last batch of a chunk may be shorter, Q7) */
  int x_per_model;      /* 0: one [B,d] batch shared by all models (expand_dims=True); 1: [M,B,d] */
  float lr, beta1, beta2, eps, eps_root; /* torchopt.adam hyper-parameters */
  int adam_count_mode;  /* sce_adam_count */
  int fwd_passes;       /* 3: split operands (~fp32 accuracy; default), 1: the 16-bit plane only (bf16 or fp16) */
  int bwd_passes;       /* same for the three backward GEMMs */
  float norm_floor;     /* clamp floor of the row norms: 1e-8 (SAE variants); <= 0 disables it (TopK) */
  int arith;            /* enum sce_arith; 0 = AUTO */
  int topk_k_max;       /* SCE_TOPK: the largest buffers["sparsity"] of the ensemble (1..256) enables the k-sparse decode /
                           code-gradient kernels; 0 = unknown: dense GEMMs on the k-sparse code, as the reference does */
  int centering;        /* FunctionalTiedSAE.center (sae_ensemble.py:126-128) applied to the batch on the device:
                           x_c[m] = (rot[m] (x - trans[m])) * scale[m]. 0 = off (identity centring); 1 = the batch is one
                           [B,d] array shared by all models; 2 = [M,B,d]. Needs x_per_model = 1 (the centred batch differs per
                           model) and the three center_* buffers. */
} sce_desc;

/* Device pointers owned by the caller; all fp32 unless noted. Unused ones are NULL. */
typedef struct sce_buffers {
  float* encoder;       /* [M,n,d]  params["encoder"] (tied/untied) or params["dict"] (topk) */
  float* encoder_bias;  /* [M,n]    params["encoder_bias"]; NULL for topk */
  float* decoder;       /* [M,n,d]  params["decoder"]; untied only */
  float* encoder_m;     /* Adam first moment of encoder, same shape; likewise below */
  float* encoder_v;
  float* bias_m;
  float* bias_v;
  float* decoder_m;
  float* decoder_v;
  const float* l1_alpha;          /* [M]   buffers["l1_alpha"]; NULL = 0 (topk) */
  const float* bias_decay;        /* [M]   buffers["bias_decay"]; NULL = 0 */
  const unsigned char* coef_mask; /* [M,n] buffers["coef_mask"] (1 = unused coefficient) or NULL */
  const long long* sparsity;      /* [M]   buffers["sparsity"] (topk k) or NULL. Every k in [1, n], and, when
                                     desc.topk_k_max is in 1..256 (the plan keeps k-sparse lists), k <= topk_k_max;
                                     read by sce_prepare, which rejects other values */
  void* workspace;                /* >= sce_workspace_bytes(desc), 1024-byte aligned */
  size_t workspace_bytes;
  const float* center_trans;      /* [M,d]   buffers["center_trans"]  (desc.centering != 0; else NULL) */
  const float* center_rot;        /* [M,d,d] buffers["center_rot"]    */
  const float* center_scale;      /* [M,d]   buffers["center_scale"]  */
} sce_buffers;

typedef struct sce_plan sce_plan;

/* Loss columns written by sce_step: out_losses[m*SCE_LOSS_COLS + k]. */
enum { SCE_LOSS_TOTAL = 0, SCE_LOSS_RECONSTRUCTION = 1, SCE_LOSS_L1 = 2, SCE_LOSS_BIAS_DECAY = 3, SCE_LOSS_COLS = 4 };

int sce_version(void);
const char* sce_last_error(void);

/* Bytes of device scratch a plan needs (operand planes — 4 bytes per element — of the dictionary, the batch, the code, the
 * residual and the code gradient; fp32 weight gradients; reduction partials). */
size_t sce_workspace_bytes(const sce_desc* desc);

/* Builds the TMA descriptors and kernel launch plan. Does not touch device memory. */
int sce_plan_create(const sce_desc* desc, const sce_buffers* buffers, sce_plan** out_plan);
int sce_plan_destroy(sce_plan* plan);

/* (Re)derive the normalised operand planes of the dictionaries from the fp32 parameters. Must be
 * called once before the first step and again whenever the caller modified the parameters itself.
 * SCE_TOPK: also re-reads buffers.sparsity (the k of each model) and returns SCE_ERR_INVALID if a k is < 1 or > n, or,
 * on a plan that keeps k-sparse lists, > desc.topk_k_max: the lists hold at most that many entries per row, so a larger
 * k needs a new plan. Until it succeeds the plan must not run. */
int sce_prepare(sce_plan* plan, void* stream);

/* One optimisation step for all M models on one batch == FunctionalEnsemble.step_batch (ensemble.py:175-193):
 * forward, losses, backward, Adam, in-place parameter update.
 *   x          device fp32, [B,d] (x_per_model = 0) or [M,B,d]
 *   out_losses device fp32 [M, SCE_LOSS_COLS]
 *   out_nnz    device fp32 [M]: mean over the batch of count_nonzero(c, -1)  (big_sweep.py:171)            */
int sce_step(sce_plan* plan, const float* x, int B, float* out_losses, float* out_nnz, void* stream);

/* Same step, fed from HOST memory the way the reference loop feeds it (big_sweep.py:168): copies `x_host`
 * (pinned or pageable fp32) to the device, steps, copies the [M,SCE_LOSS_COLS] losses and [M] nnz back, and
 * synchronises the stream before returning. */
int sce_step_host(sce_plan* plan, const float* x_host, int B, float* out_losses_host, float* out_nnz_host,
                  void* stream);

/* Forward only (evaluation; LearnedDict.predict semantics on already-centred inputs): writes x_hat
 * [M,B,d] fp32 if non-NULL and the same losses / nnz as sce_step, without touching parameters. */
int sce_forward(sce_plan* plan, const float* x, int B, float* x_hat, float* out_losses, float* out_nnz,
                void* stream);

/* Materialise the fp32 code tensor aux["c"] [M,B,n] of the most recent step/forward (compat path for callers
 * that really want the dense tensor the reference returns, ensemble.py:193). */
int sce_read_code(sce_plan* plan, int B, float* out_code, void* stream);

/* Materialise the fp32 parameter gradients of the most recent sce_grads call (parity tests). */
int sce_grads(sce_plan* plan, const float* x, int B, float* d_encoder, float* d_bias, float* d_decoder,
              float* out_losses, float* out_nnz, void* stream);

/* Split a row-gathered, optionally mean-centred batch out of a resident activation chunk:
 *   out[r,:] = float(chunk[idx[r],:]) - sub[:]      chunk fp16 or fp32 [N,d]; idx int64 [B] or NULL (identity)
 * (big_sweep.py:168 `dataset[batch_idxs]`, :359-364 centring) */
int sce_gather_rows(const void* chunk, int chunk_is_half, long long n_rows, int d, const long long* idx, int B,
                    const float* sub, float* out, void* stream);

/* Per-phase device timing of sce_step, measured with CUDA events recorded on the caller's stream between the
 * kernels of a step (bench.py's roofline). Between sce_profile_begin and sce_profile_end up to 64 steps are
 * recorded; sce_profile_end synchronises and returns the summed milliseconds of each phase. */
enum {
  SCE_PHASE_SPLIT = 0,  /* batch -> (hi, lo) */
  SCE_PHASE_ENCODE = 1, /* encode GEMM (+ top-k selection) */
  SCE_PHASE_DECODE = 2, /* decode GEMM + residual */
  SCE_PHASE_LOSSES = 3, /* bias norm + loss finalisation */
  SCE_PHASE_DCODE = 4,  /* code-gradient GEMM */
  SCE_PHASE_DW = 5,     /* weight-gradient GEMM(s) */
  SCE_PHASE_ADAM = 6,   /* Jacobian + Adam + renormalise + re-split, bias Adam */
  SCE_PHASE_COUNT = 7
};
int sce_profile_begin(sce_plan* plan);
int sce_profile_end(sce_plan* plan, float* phase_ms /*[SCE_PHASE_COUNT]*/, int* steps_recorded);

/* Optimiser step counter (number of sce_step calls so far); settable so a resumed run keeps the bias correction
 * of SCE_ADAM_STANDARD continuous. */
long long sce_get_step_count(const sce_plan* plan);
int sce_set_step_count(sce_plan* plan, long long steps_taken);

/* Number of kernels the most recent sce_step / sce_forward on this plan launched. */
int sce_last_launch_count(const sce_plan* plan);

/* F16F8 plans: the largest |x| over every batch fed since the last sce_prepare (NaN if a batch held one), read back
 * with one 4-byte copy and a stream synchronise — a monitor for the fp16 range the arithmetic assumes (values beyond
 * 65504 become inf/NaN in the losses, magnitudes far below 1e-3 lose relative precision: use SCE_ARITH_BF16X3 for
 * such data). BF16X3 plans report 0. */
int sce_input_absmax(sce_plan* plan, float* out_host, void* stream);

/* Health of the run. *bad_out = 1 when some step since the last sce_prepare / sce_clear_health saw a batch the fp16
 * operand plane cannot hold (F16F8: |x| >= 65520 or NaN) or produced a non-finite loss. From that step on the Adam
 * kernels leave parameters, moments and operand planes UNTOUCHED (the update is skipped on the device, so a bad chunk
 * cannot write NaN into the caller's tensors before the host looks); the caller decides: raise, or rebuild the plan
 * with SCE_ARITH_BF16X3. *absmax_out as sce_input_absmax. One 512-byte copy and a stream synchronise. */
int sce_health(sce_plan* plan, int* bad_out, float* absmax_out, void* stream);
int sce_clear_health(sce_plan* plan, void* stream);

/* Per-feature activation counts of the most recent step / forward: counts[m][j] += number of the B rows whose code
 * c[m, r, j] is non-zero (device int32 [M, n], ACCUMULATED so that a held-out set can be streamed through in batches).
 * This is the reference's `(c != 0).sum(0)` (standard_metrics.py:441-454, "features ever active" = count > threshold)
 * and, divided by the rows, its `(c != 0).float().mean(0)` (:305-308). Reads only the activity-mask plane the encode
 * epilogue / top-k selection wrote (B/8 bytes per feature chunk): the dense code is never materialised. */
int sce_active_counts(sce_plan* plan, int B, int* counts, void* stream);

/* The arithmetic the plan resolved to: SCE_ARITH_BF16X3 or SCE_ARITH_F16F8. */
int sce_plan_arith(const sce_plan* plan);

#ifdef __cplusplus
}
#endif
#endif /* SCE_H_ */
