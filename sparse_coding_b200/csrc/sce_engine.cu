// sce_engine.cu — libsce.so: the C ABI of include/sce.h on top of the tcgen05 GEMM core and the
// streaming kernels. One `sce_plan` = one stacked ensemble (FunctionalEnsemble, autoencoders/ensemble.py:68-97).
//
// One training step (tied variant; untied and top-k differ as noted; "(hi, lo)" stands for the operand planes of the
// plan's arithmetic: fp16 + two E5M2 planes with f16f8, a bf16 pair with bf16x3) is
//   split_rows      x -> (x_hi, x_lo)  [+ residual-plane flag, input range monitor]
//   GEMM encode     z = x W^T (+b) -> relu -> (c_hi, c_lo), activity masks, sum|c|, nnz   [M x B x n, K = d]
//   GEMM decode     x^ = c W -> r = x^ - x, sum r^2, g = 2r/(Bd) -> (g_hi, g_lo)  [M x B x d, K = n]
//   GEMM dcode      dz = (g W^T + alpha/B [c>0]) [z>=0] -> (dz_hi, dz_lo), db partials
//   GEMM dW         dW = dz^T x + c^T g                                            [M x n x d, K = 2B]
//   bias_norm, finalize (losses), dict_rows<ADAM> (Jacobian + Adam + renormalise + re-split), bias<ADAM>
// Top-k variant: the encode GEMM stores fp32 scores; topk_select2_kernel keeps k per row; with the k-sparse path
// (sce_topk.cuh) decode and dcode are a gather kernel over the k selected dictionary rows instead of two dense GEMMs.
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <vector>
#include <new>

#include "../../include/sce.h"
#include "sce_epilogues.cuh"
#include "sce_gemm.cuh"
#include "sce_kernels.cuh"
#include "sce_topk.cuh"
#include "sce_tmap.h"

using namespace sce;

// ------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";
static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
#define CUDA_TRY(x)                                                                            \
  do {                                                                                         \
    cudaError_t e_ = (x);                                                                      \
    if (e_ != cudaSuccess) return fail(SCE_ERR_CUDA, "%s failed: %s", #x, cudaGetErrorString(e_)); \
  } while (0)

// ------------------------------------------------------------------------------------------------
// plan
// ------------------------------------------------------------------------------------------------
struct GemmMaps {  // tensor maps of one GEMM for one batch size (x8: third plane of the f16f8 arithmetic)
  CUtensorMap a_hi[kMaxSets], a_lo[kMaxSets], b_hi[kMaxSets], b_lo[kMaxSets];
  CUtensorMap a_x8[kMaxSets], b_x8[kMaxSets];
};
struct BatchMaps {
  GemmMaps encode, decode, dcode, dw_enc, dw_dec;
  GemmMaps center;             // centring: A = (x - trans) planes [M,B,d], B = rot planes [M,d,d], both K-major
  CUtensorMap st_c_hi, st_c_lo, st_c_x8, st_dz_hi, st_dz_lo, st_dz_x8;  // epilogue TMA-store maps
  CUtensorMap st_scores;                                                // top-k: fp32 scores
  cudaGraphExec_t graph;       // captured step for this batch size (launch-bound shapes), or nullptr
  int graph_launches, eager_steps;
};

struct sce_plan {
  sce_desc d;
  sce_buffers b;
  int sms;
  int device;  // CUDA device the plan was created on (the caller keeps it current for every call)
  int xm;  // number of distinct input batches (1 shared, or M)
  // workspace carve-up
  // Operand planes. bf16x3: hi, lo = bf16 planes (2 B / element each), x8 unused. f16f8: hi = fp16 plane, lo =
  // e5m2 plane of the values, x8 = e5m2 plane of the scaled residuals (1 B / element each): 4 B / element either way.
  int arith;                      // kArithBf16x3 or kArithF16F8 (resolved from desc.arith / env SCE_ARITH / the shape)
  float* x_stage;                 // [xm, Bmax, d] staging for host-fed steps
  __nv_bfloat16 *x_hi, *x_lo;     // [xm, Bmax, d]
  __nv_bfloat16 *wenc_hi, *wenc_lo, *wdec_hi, *wdec_lo;  // [M, n, d] (tied: dec aliases enc)
  __nv_bfloat16 *c_hi, *c_lo;     // [M, Bmax, n]
  __nv_bfloat16 *g_hi, *g_lo;     // [M, Bmax, d]
  __nv_bfloat16 *dz_hi, *dz_lo;   // [M, Bmax, n]   (top-k: fp32 scores alias these planes)
  uint8_t *x_x8, *wenc_x8, *wdec_x8, *c_x8, *g_x8, *dz_x8;
  __nv_bfloat16 *rot_hi, *rot_lo;  // centring: operand planes of buffers["center_rot"] [M, d, d]
  uint8_t* rot_x8;
  float* x_centered;              // centring: the centred batch [M, B, d] (B, not Bmax, rows per model: what a caller's [M,B,d] looks like)
  float* scores;                  // top-k: fp32 scores [M, Bmax, n] of the encode GEMM
  int* tk_models;                 // top-k gather kernel: the models sorted into k classes (device copy of tk_group_models)
  int tk_groups, tk_group_off[5], tk_group_krows[4];   // classes: models [off[g], off[g+1]) need at most krows[g] rows
  uint32_t* tk_cmax;              // top-k: largest key per 32-column chunk of the scores [M, Bmax, n_chunks] (EpiScoresTma)
  int topk_cmax;                  // 1: the selection works from the chunk maxima (SCE_TOPK_CMAX=0 turns it off)
  int *tk_col, *tk_cnt;           // top-k lists (TopkLists): selected columns [M, Bmax, kmax], entries per row [M, Bmax]
  float *tk_val, *tk_dots;        // their values [M, Bmax, kmax]; per-slice shares of g . W_j [M, Bmax, kmax, slices]
  float* wn_f32;                  // top-k: fp32 copy of the normalised dictionary [M, n, d] the gather kernel reads
  int tk_slices;                  // slices of the activation width topk_sparse_kernel runs per row
  int tk_kmax;                    // list capacity per row (desc.topk_k_max rounded up to 8; 0: no lists)
  int topk_sparse;                // 1: decode / dcode of the top-k variant run as the k-sparse gather kernels
  uint32_t *act_pos, *act_zero;   // activity masks [M][ceil(n/32)][Bmax]: bit 31-j of a word = column 32*chunk + j (ActMask)
  uint32_t* res_flags;            // [0]: the batch has a non-zero residual plane (f16f8; written by the batch split)
  float *dw_enc, *dw_dec;         // [M, n, d]
  float *part_enc, *part_dec, *db_part, *bnorm, *l1_over_b, *loss_stage, *nnz_stage;
  int tiles_mB_max;
  std::map<int, BatchMaps*>* maps;
  cudaStream_t cap_stream;  // private stream the step is captured on
  int dcode_passes, dw_passes;  // tensor passes of the two backward GEMMs (default: desc.bwd_passes)
  int use_graph;     // 1: replay the step as a CUDA graph (launch-bound shapes; env SCE_GRAPH overrides)
  int split_decode;  // 1: separate TMEM accumulators for hi*hi and the cross terms in the decode GEMM (default)
  int pair_encode, pair_decode, pair_dcode, pair_dw;  // 1: run that GEMM on CTA pairs (cta_group::2, 256-row tiles)
  int bk_encode, bk_decode, bk_dcode;  // K block (64: 128-byte swizzle, 32: 64-byte swizzle) of the K-major GEMMs
  int dw_collector;  // NSUB = 2 tiles: A slice kept in the tensor core's collector across the two column halves (SCE_TUNE_DW_COLL)
  int dec_nsub2;     // experiment: decode with 256 x 512 tiles (SCE_TUNE_DEC_NSUB2)
  int dw_nsub2;      // f16f8 weight gradient: 256 x 512 tiles sharing one A tile (env SCE_TUNE_DW_NSUB2 = 0 switches it off)
  int last_launches;
  long long step;  // number of optimiser steps taken
  // optional per-phase device timing (sce_profile_*): events bracket each phase of a step
  bool prof_on;
  int prof_steps;                          // steps recorded since sce_profile_begin
  cudaEvent_t* prof_ev;                    // [kProfMaxSteps][SCE_PHASE_COUNT + 1]
};

constexpr int kProfMaxSteps = 64;
static inline void prof_mark(sce_plan* p, int idx, cudaStream_t st) {
  if (p->prof_on && p->prof_steps < kProfMaxSteps)
    cudaEventRecord(p->prof_ev[p->prof_steps * (SCE_PHASE_COUNT + 1) + idx], st);
}

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct Carve {
  uint8_t* base;
  size_t off;
  template <class T>
  T* take(size_t count) {
    off = align_up(off, 1024);
    T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += count * sizeof(T);
    return p;
  }
};

static int validate(const sce_desc* d) {
  if (!d) return fail(SCE_ERR_INVALID, "desc is NULL");
  if (d->variant < SCE_TIED || d->variant > SCE_TOPK) return fail(SCE_ERR_INVALID, "unknown variant %d", d->variant);
  if (d->n_models < 1 || d->batch_max < 1) return fail(SCE_ERR_INVALID, "n_models and batch_max must be >= 1");
  if (d->d < 8 || d->d % 8 || d->n < 8 || d->n % 8)
    return fail(SCE_ERR_INVALID, "d (%d) and n (%d) must be positive multiples of 8", d->d, d->n);
  if (d->d > 8192) return fail(SCE_ERR_INVALID, "d = %d > 8192 is not supported by the row kernels", d->d);
  if ((d->fwd_passes != 1 && d->fwd_passes != 3) || (d->bwd_passes != 1 && d->bwd_passes != 3))
    return fail(SCE_ERR_INVALID, "fwd_passes / bwd_passes must be 1 or 3");
  if (d->centering < 0 || d->centering > 2) return fail(SCE_ERR_INVALID, "centering must be 0, 1 or 2");
  if (d->centering && !d->x_per_model) return fail(SCE_ERR_INVALID, "centering needs x_per_model = 1 (the centred batch differs per model)");
  if (d->arith < SCE_ARITH_AUTO || d->arith > SCE_ARITH_F16F8) return fail(SCE_ERR_INVALID, "unknown arith %d", d->arith);
  if (d->arith == SCE_ARITH_F16F8 && (d->d % 16 || d->n % 16))
    return fail(SCE_ERR_INVALID, "arith = F16F8 needs d (%d) and n (%d) to be multiples of 16 (TMA pitch of the 8-bit planes)",
                d->d, d->n);
  return SCE_OK;
}

// desc.arith -> kArithBf16x3 / kArithF16F8. AUTO: f16f8 where the 8-bit planes can be addressed by TMA
// (row pitches of 16 bytes), bf16x3 otherwise; the environment may pin AUTO to one of them (A/B runs).
static int resolve_arith(const sce_desc& d) {
  if (d.arith == SCE_ARITH_BF16X3) return kArithBf16x3;
  if (d.arith == SCE_ARITH_F16F8) return kArithF16F8;
  const bool shape_ok = d.d % 16 == 0 && d.n % 16 == 0;
  if (const char* v = getenv("SCE_ARITH")) {
    if (!strcmp(v, "bf16x3")) return kArithBf16x3;
    if (!strcmp(v, "f16f8") && shape_ok) return kArithF16F8;
  }
  return shape_ok ? kArithF16F8 : kArithBf16x3;
}

// capacity per row of the top-k lists: the largest k of the ensemble (desc.topk_k_max, supplied by the host mirror, which
// knows buffers["sparsity"]) rounded up to 8; 0 = unknown or too large for the gather kernel -> dense path, no lists
static size_t topk_kmax(const sce_desc& d) {
  if (d.variant != SCE_TOPK || d.topk_k_max < 1 || d.topk_k_max > 256) return 0;
  return (size_t)(d.topk_k_max + 7) / 8 * 8;
}
// topk_sparse_kernel: dynamic shared memory for `slices` slices of the activation width (see there), and the slice
// count a plan uses: the smallest of 2, 4, 8 whose slice fits (two blocks per SM); 0 when none does (the plan then runs
// the dense GEMMs)
constexpr int kTopkMaxSlices = 8;
static size_t topk_sparse_smem(const sce_desc& d, size_t krows, int slices) {
  const size_t ds = d.d / slices;
  return krows * ds * sizeof(float) + 9 * ds * sizeof(float) + krows * 8 + 128;
}
static int topk_slices(const sce_desc& d, size_t kmax) {
  int best = 0;
  for (int s = 2; s <= kTopkMaxSlices; s *= 2) {
    if (d.d % (4 * s) || d.d / s > 512) continue;
    const size_t b = topk_sparse_smem(d, kmax, s);
    if (b <= 112 * 1024) return s;   // fewest slices that fit: the kernel's time goes with the number of blocks
  }
  return best;
}

// Carves the workspace; with base == nullptr only measures it.
static size_t carve(sce_plan* p, const sce_desc& d, uint8_t* base) {
  Carve c{base, 0};
  const size_t M = d.n_models, B = d.batch_max, n = d.n, dd = d.d;
  const size_t xm = d.x_per_model ? M : 1;
  const size_t tiles_mB = (B + kBM - 1) / kBM;
  const size_t tiles_nN = (n + 127) / 128;  // upper bound over the BN choices (BN >= 128)
  const size_t tiles_nD = (dd + 127) / 128;
  const bool f8 = resolve_arith(d) == kArithF16F8;
  // the planes of one operand tensor: 16-bit, then (bf16x3) a second 16-bit plane or (f16f8) two 8-bit planes
  auto planes = [&](size_t count, __nv_bfloat16*& hi, __nv_bfloat16*& lo, uint8_t*& x8) {
    hi = c.take<__nv_bfloat16>(count);
    if (f8) {
      lo = reinterpret_cast<__nv_bfloat16*>(c.take<uint8_t>(count));
      x8 = c.take<uint8_t>(count);
    } else {
      lo = c.take<__nv_bfloat16>(count);
      x8 = nullptr;
    }
  };
  auto X = c.take<float>(xm * B * dd);
  __nv_bfloat16 *xh, *xl, *weh, *wel, *ch, *cl, *gh, *gl;
  uint8_t *x8, *we8, *c8, *g8;
  planes(xm * B * dd, xh, xl, x8);
  planes(M * n * dd, weh, wel, we8);
  __nv_bfloat16 *wdh = weh, *wdl = wel;
  uint8_t* wd8 = we8;
  if (d.variant == SCE_UNTIED) planes(M * n * dd, wdh, wdl, wd8);
  planes(M * B * n, ch, cl, c8);
  planes(M * B * dd, gh, gl, g8);
  auto dzh = c.take<__nv_bfloat16>(2 * M * B * n);  // all planes contiguous, 4 B / element: the top-k scores alias them
  auto dwe = c.take<float>(M * n * dd);
  float* dwd = dwe;
  if (d.variant == SCE_UNTIED) dwd = c.take<float>(M * n * dd);
  const size_t enc_parts = d.variant == SCE_TOPK ? B : tiles_mB * 8 * tiles_nN;
  auto pe = c.take<float>(M * enc_parts * 2);
  const size_t dec_parts = tiles_mB * 8 * tiles_nD;   // top-k: up to kTopkMaxSlices partials per row from the gather kernel
  auto pd = c.take<float>(M * (d.variant == SCE_TOPK && dec_parts < kTopkMaxSlices * B ? kTopkMaxSlices * B : dec_parts));
  auto dbp = c.take<float>(M * tiles_mB * 4 * n);
  auto bn = c.take<float>(M);
  auto lob = c.take<float>(M);
  auto ls = c.take<float>(M * 4);
  auto ns = c.take<float>(M);
  const size_t n_chunks = (n + 31) / 32;
  auto apos = c.take<uint32_t>(M * n_chunks * B);
  auto azero = c.take<uint32_t>(M * n_chunks * B);
  // top-k: scores of their own (the code-gradient planes must keep their scattered zeros) and the k-sparse lists
  const size_t kmax = topk_kmax(d);
  float* sc = nullptr;
  int *tkc = nullptr, *tkn = nullptr, *tkm = nullptr;
  float *tkv = nullptr, *tkd = nullptr, *wnf = nullptr;
  uint32_t* tcm = nullptr;
  if (d.variant == SCE_TOPK) {
    sc = c.take<float>(M * B * n);
    tcm = c.take<uint32_t>(M * B * n_chunks);
    if (kmax) {
      tkc = c.take<int>(M * B * kmax);
      tkv = c.take<float>(M * B * kmax);
      tkn = c.take<int>(M * B);
      tkm = c.take<int>(M);
      tkd = c.take<float>(M * B * kmax * kTopkMaxSlices);
      wnf = c.take<float>(M * n * dd);
    }
  }
  __nv_bfloat16 *roth = nullptr, *rotl = nullptr;
  uint8_t* rot8 = nullptr;
  float* xcen = nullptr;
  if (d.centering) {
    planes(M * dd * dd, roth, rotl, rot8);
    xcen = c.take<float>(M * B * dd);
  }
  auto rf = c.take<uint32_t>(kFlagWords);   // [0] residual flag, [kAbsmaxWord] input range monitor, [kBadWord] health (separate 128-byte lines)
  if (p) {
    p->x_stage = X;
    p->x_hi = xh;
    p->x_lo = xl;
    p->wenc_hi = weh;
    p->wenc_lo = wel;
    p->wdec_hi = wdh;
    p->wdec_lo = wdl;
    p->c_hi = ch;
    p->c_lo = cl;
    p->g_hi = gh;
    p->g_lo = gl;
    p->dz_hi = dzh;
    p->dz_lo = dzh + M * B * n;
    p->dz_x8 = f8 ? reinterpret_cast<uint8_t*>(dzh) + 3 * M * B * n : nullptr;
    p->x_x8 = x8;
    p->wenc_x8 = we8;
    p->wdec_x8 = wd8;
    p->c_x8 = c8;
    p->g_x8 = g8;
    p->dw_enc = dwe;
    p->dw_dec = dwd;
    p->part_enc = pe;
    p->part_dec = pd;
    p->db_part = dbp;
    p->bnorm = bn;
    p->l1_over_b = lob;
    p->loss_stage = ls;
    p->nnz_stage = ns;
    p->res_flags = rf;
    p->rot_hi = roth;
    p->rot_lo = rotl;
    p->rot_x8 = rot8;
    p->x_centered = xcen;
    p->scores = sc;
    p->tk_cmax = tcm;
    p->tk_models = tkm;
    p->tk_col = tkc;
    p->tk_val = tkv;
    p->tk_cnt = tkn;
    p->tk_dots = tkd;
    p->wn_f32 = wnf;
    p->tk_kmax = (int)kmax;
    p->act_pos = apos;
    p->act_zero = azero;
    p->tiles_mB_max = (int)tiles_mB;
  }
  return align_up(c.off, 1024);
}

// ------------------------------------------------------------------------------------------------
// tensor maps for one batch size
// ------------------------------------------------------------------------------------------------
static int bn_for(int N) { return N > 128 ? 256 : 128; }
// a CTA pair needs at least two 128-row blocks of output
static bool use_pair(int flag, int rows) { return flag && rows > kBM; }
constexpr int kBkDw = 32;  // K block of the MN-major weight-gradient GEMM
// K block of the GEMMs with K-major operands: 32 (64-byte swizzle, 4 stages of 48 KB at BN = 256) keeps three
// stages in flight behind the one being multiplied; 64 (128-byte swizzle) only has room for two stages.
// Chosen per GEMM (plan fields bk_encode / bk_decode / bk_dcode; env SCE_TUNE_BK_{ENCODE,DECODE,DCODE} overrides):
// measured on B200 (profiles/r01f_bk_tuning.txt) the deeper pipeline wins where the A operand streams from HBM
// (decode: the code tensor) and loses where both operands are L2-resident (encode, dcode: twice the TMA requests).
static int tune_bk(const char* env, int dflt) {
  const char* v = getenv(env);
  if (!v) return dflt;
  const int k = atoi(v);
  return (k == 32 || k == 64) ? k : dflt;
}
static int tune_flag(const char* env, int dflt) {
  const char* v = getenv(env);
  return v ? (atoi(v) != 0) : dflt;
}
static CUtensorMapSwizzle swizzle_for_bk(int bk) {
  return bk == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B;
}

static CUtensorMapSwizzle swizzle8_for_bk(int bk) {  // K-major 8-bit tiles: rows of bk bytes
  return bk == 32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_64B;
}
constexpr int kBkF8 = 64;  // K block of every GEMM in the f16f8 arithmetic

// The planes of one operand [models][rows][cols] (cols contiguous, `mpitch` elements between models) as GEMM operand
// maps. kmajor_bk != 0: K-major tiles [box_rows][kmajor_bk]; else MN-major tiles of `box_rows` k-rows by 64 (16-bit)
// / 128 (8-bit) contiguous elements.
static bool operand_maps(int arith, CUtensorMap* hi, CUtensorMap* lo, CUtensorMap* x8, const void* phi, const void* plo,
                         const void* px8, uint64_t models, uint64_t rows, uint64_t cols, uint64_t mpitch,
                         uint32_t box_rows, int kmajor_bk) {
  bool ok;
  if (kmajor_bk) {
    ok = make_tmap_bf16_box(hi, phi, models, rows, cols, cols, mpitch, kmajor_bk, box_rows, swizzle_for_bk(kmajor_bk));
    if (arith == kArithF16F8)
      ok = ok && make_tmap_u8_box(lo, plo, models, rows, cols, cols, mpitch, kmajor_bk, box_rows, swizzle8_for_bk(kmajor_bk)) &&
           make_tmap_u8_box(x8, px8, models, rows, cols, cols, mpitch, kmajor_bk, box_rows, swizzle8_for_bk(kmajor_bk));
    else
      ok = ok && make_tmap_bf16_box(lo, plo, models, rows, cols, cols, mpitch, kmajor_bk, box_rows, swizzle_for_bk(kmajor_bk));
  } else {
    ok = make_tmap_bf16(hi, phi, models, rows, cols, cols, mpitch, box_rows);
    if (arith == kArithF16F8)
      ok = ok && make_tmap_u8_box(lo, plo, models, rows, cols, cols, mpitch, 128, box_rows, CU_TENSOR_MAP_SWIZZLE_128B) &&
           make_tmap_u8_box(x8, px8, models, rows, cols, cols, mpitch, 128, box_rows, CU_TENSOR_MAP_SWIZZLE_128B);
    else
      ok = ok && make_tmap_bf16(lo, plo, models, rows, cols, cols, mpitch, box_rows);
  }
  return ok;
}

static int build_maps(sce_plan* p, int B, BatchMaps** out) {
  auto it = p->maps->find(B);
  if (it != p->maps->end()) {
    *out = it->second;
    return SCE_OK;
  }
  BatchMaps* m = new (std::nothrow) BatchMaps;
  if (!m) return fail(SCE_ERR_INVALID, "out of host memory");
  memset(m, 0, sizeof(*m));
  const sce_desc& d = p->d;
  const uint64_t M = d.n_models, n = d.n, dd = d.d, xm = p->xm, Bm = d.batch_max;
  // NOTE: activations are laid out with the plan's batch_max pitch between models; only `B` rows are
  // visible through the map, so rows >= B read as zero (TMA out-of-bounds fill).
  const int ar = p->arith;
  const bool f8 = ar == kArithF16F8;
  const int bk_enc = f8 ? kBkF8 : p->bk_encode, bk_dec = f8 ? kBkF8 : p->bk_decode, bk_dco = f8 ? kBkF8 : p->bk_dcode;
  const int bk_dw = f8 ? kBkF8 : kBkDw;
  // the f16f8 kernels run narrow outputs (<= 128 columns) on single CTAs: an MN-major 8-bit B tile is 128 wide
  auto pair_ok = [&](int flag, int rows, int out_cols) { return use_pair(flag, rows) && !(f8 && out_cols <= 128); };
  struct Pl { const void *hi, *lo, *x8; };
  const Pl X{p->x_hi, p->x_lo, p->x_x8}, WE{p->wenc_hi, p->wenc_lo, p->wenc_x8}, WD{p->wdec_hi, p->wdec_lo, p->wdec_x8},
      C{p->c_hi, p->c_lo, p->c_x8}, G{p->g_hi, p->g_lo, p->g_x8}, DZ{p->dz_hi, p->dz_lo, p->dz_x8};
  // activations [models][B of batch_max][cols]: K-major A tiles [128 rows][bk] / MN-major tiles of bk_dw batch rows
  auto actk = [&](GemmMaps& g, int set, const Pl& P, uint64_t models, uint64_t cols, int bk) {
    return operand_maps(ar, &g.a_hi[set], &g.a_lo[set], &g.a_x8[set], P.hi, P.lo, P.x8, models, (uint64_t)B, cols, Bm * cols, kBM, bk);
  };
  auto act_a = [&](GemmMaps& g, int set, const Pl& P, uint64_t models, uint64_t cols) {
    return operand_maps(ar, &g.a_hi[set], &g.a_lo[set], &g.a_x8[set], P.hi, P.lo, P.x8, models, (uint64_t)B, cols, Bm * cols, bk_dw, 0);
  };
  auto act_b = [&](GemmMaps& g, int set, const Pl& P, uint64_t models, uint64_t cols) {
    return operand_maps(ar, &g.b_hi[set], &g.b_lo[set], &g.b_x8[set], P.hi, P.lo, P.x8, models, (uint64_t)B, cols, Bm * cols, bk_dw, 0);
  };
  // dictionary [M][n][d] as the B operand: K-major tiles [box_rows][bk] (box_rows = the B rows ONE CTA loads), or MN-major
  auto dict_b = [&](GemmMaps& g, const Pl& P, uint32_t box_rows, int kmajor_bk) {
    return operand_maps(ar, &g.b_hi[0], &g.b_lo[0], &g.b_x8[0], P.hi, P.lo, P.x8, M, n, dd, n * dd, box_rows, kmajor_bk);
  };
  bool ok = true;
  // encode: A = x [xm,B,d] K-major, B = Wenc [M,n,d] K-major
  ok &= actk(m->encode, 0, X, xm, dd, bk_enc);
  ok &= dict_b(m->encode, WE, bn_for(d.n) / (pair_ok(p->pair_encode, B, d.n) ? 2 : 1), bk_enc);
  if (d.centering) {
    // centring: A = (x - trans) planes in the X planes (the encode A maps), B = rot [M,d,d] K-major, output d columns
    for (int t = 0; t < 1; ++t) {
      m->center.a_hi[t] = m->encode.a_hi[t];
      m->center.a_lo[t] = m->encode.a_lo[t];
      m->center.a_x8[t] = m->encode.a_x8[t];
    }
    ok &= operand_maps(ar, &m->center.b_hi[0], &m->center.b_lo[0], &m->center.b_x8[0], p->rot_hi, p->rot_lo, p->rot_x8, M, dd, dd,
                       dd * dd, bn_for(d.d) / (pair_ok(p->pair_encode, B, d.d) ? 2 : 1), bk_enc);
  }
  // decode: A = c [M,B,n] K-major, B = Wdec [M,n,d] MN-major (bk k-rows per box)
  ok &= actk(m->decode, 0, C, M, n, bk_dec);
  ok &= dict_b(m->decode, WD, bk_dec, 0);
  // dcode: A = g [M,B,d] K-major, B = Wdec K-major
  ok &= actk(m->dcode, 0, G, M, dd, bk_dco);
  ok &= dict_b(m->dcode, WD, bn_for(d.n) / (pair_ok(p->pair_dcode, B, d.n) ? 2 : 1), bk_dco);
  // weight gradients: everything MN-major, reduction over the batch rows
  if (d.variant == SCE_UNTIED) {
    ok &= act_a(m->dw_enc, 0, DZ, M, n);
    ok &= act_b(m->dw_enc, 0, X, xm, dd);
    ok &= act_a(m->dw_dec, 0, C, M, n);
    ok &= act_b(m->dw_dec, 0, G, M, dd);
  } else {
    ok &= act_a(m->dw_enc, 0, DZ, M, n);
    ok &= act_b(m->dw_enc, 0, X, xm, dd);
    ok &= act_a(m->dw_enc, 1, C, M, n);
    ok &= act_b(m->dw_enc, 1, G, M, dd);
  }
  if (f8 && SCE_EPI_PAIR) {
    // two adjacent chunks per bulk store (stage_pair_and_store): boxes of 64 columns x 32 rows, 128-byte rows
    ok &= make_tmap_bf16_box(&m->st_c_hi, p->c_hi, M, (uint64_t)B, n, n, Bm * n, 64, 32, CU_TENSOR_MAP_SWIZZLE_128B);
    ok &= make_tmap_bf16_box(&m->st_dz_hi, p->dz_hi, M, (uint64_t)B, n, n, Bm * n, 64, 32, CU_TENSOR_MAP_SWIZZLE_128B);
  } else {
    ok &= make_tmap_bf16_store32(&m->st_c_hi, p->c_hi, M, (uint64_t)B, n, Bm * n);
    ok &= make_tmap_bf16_store32(&m->st_dz_hi, p->dz_hi, M, (uint64_t)B, n, Bm * n);
  }
  if (f8) {
    auto st8 = [&](CUtensorMap* t, const void* base) {
      if (SCE_EPI_PAIR) return make_tmap_u8_box(t, base, M, (uint64_t)B, n, n, Bm * n, 64, 32, CU_TENSOR_MAP_SWIZZLE_64B);
      return make_tmap_u8_box(t, base, M, (uint64_t)B, n, n, Bm * n, 32, 32, CU_TENSOR_MAP_SWIZZLE_32B);
    };
    ok &= st8(&m->st_c_lo, p->c_lo) && st8(&m->st_c_x8, p->c_x8) && st8(&m->st_dz_lo, p->dz_lo) && st8(&m->st_dz_x8, p->dz_x8);
  } else {
    ok &= make_tmap_bf16_store32(&m->st_c_lo, p->c_lo, M, (uint64_t)B, n, Bm * n);
    ok &= make_tmap_bf16_store32(&m->st_dz_lo, p->dz_lo, M, (uint64_t)B, n, Bm * n);
  }
  if (d.variant == SCE_TOPK) ok &= make_tmap_f32_store32(&m->st_scores, p->scores, M, (uint64_t)B, n, Bm * n);
  if (!ok) {
    delete m;
    return fail(SCE_ERR_CUDA, "cuTensorMapEncodeTiled failed (B=%d, M=%d, n=%d, d=%d)", B, d.n_models, d.n, d.d);
  }
  (*p->maps)[B] = m;
  *out = m;
  return SCE_OK;
}

// ------------------------------------------------------------------------------------------------
// GEMM launcher
// ------------------------------------------------------------------------------------------------
// device flags "this operand's residual plane is all zeros" (f16f8; GemmParams::a_res_flag), nullptr = unknown
struct ResFlags {
  const uint32_t* a[kMaxSets] = {nullptr, nullptr};
  const uint32_t* b[kMaxSets] = {nullptr, nullptr};
};

template <class Epi, int BN, int BK, bool A_MN, bool B_MN, int STAGES, bool SPLIT_ACC = false, bool CTA2 = false,
          int ARITH = kArithBf16x3, int NSUB = 1>
static int launch_gemm_t(const sce_plan* p, const GemmMaps& maps, int nsets, const int* a_batched,
                         const int* b_batched, int k_total, int passes, int m_total, int n_total,
                         const typename Epi::Params& epi, cudaStream_t st, const ResFlags& rf = ResFlags()) {
  using SM = GemmSmem<BN, BK, A_MN, B_MN, STAGES, Epi::kWarpStageBytes, CTA2, ARITH, NSUB>;
  auto kern = gemm_split_kernel<Epi, BN, BK, A_MN, B_MN, STAGES, SPLIT_ACC, CTA2, ARITH, NSUB>;
  // the opt-in to > 48 KB of dynamic shared memory is per device: remember which devices have it
  static bool configured[64] = {};
  if (p->device < 0 || p->device >= 64 || !configured[p->device]) {
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SM::kBytes));
    if (p->device >= 0 && p->device < 64) configured[p->device] = true;
  }
  GemmParams<typename Epi::Params> gp;
  memset(&gp, 0, sizeof(gp));
  for (int s = 0; s < nsets; ++s) {
    gp.a_hi[s] = maps.a_hi[s];
    gp.a_lo[s] = maps.a_lo[s];
    gp.b_hi[s] = maps.b_hi[s];
    gp.b_lo[s] = maps.b_lo[s];
    gp.a_x8[s] = maps.a_x8[s];
    gp.b_x8[s] = maps.b_x8[s];
    gp.a_batched[s] = a_batched[s];
    gp.b_batched[s] = b_batched[s];
    gp.a_res_flag[s] = rf.a[s];
    gp.b_res_flag[s] = rf.b[s];
  }
  gp.nsets = nsets;
  gp.k_total = k_total;
  gp.passes = passes;
  gp.n_models = p->d.n_models;
  gp.m_total = m_total;
  gp.n_total = n_total;
  constexpr int kTileRows = CTA2 ? 2 * kBM : kBM;   // a CTA pair owns 256-row tiles
  gp.tiles_m = (m_total + kTileRows - 1) / kTileRows;
  gp.tiles_n = (n_total + NSUB * BN - 1) / (NSUB * BN);
  gp.epi = epi;
  gp.a_collector = p->dw_collector;
  const int units = CTA2 ? p->sms / 2 : p->sms;     // persistent: one CTA (or CTA pair) per SM (pair)
  int tiles = gp.n_models * gp.tiles_m * gp.tiles_n;
  if constexpr (NSUB == 2) {
    // double-width tiles halve the tile count; where that leaves the last wave mostly empty, its row blocks run as
    // single-width tiles instead (half the time each): cost in single-width tile times, per CTA (pair)
    if (gp.tiles_n == 1) {
      const int rows = gp.n_models * gp.tiles_m, rem = rows % units;
      const int cost_wide = 2 * ((rows + units - 1) / units);
      const int cost_mixed = 2 * (rows / units) + (2 * rem + units - 1) / units;
      if (rem > 0 && cost_mixed < cost_wide) {
        gp.tail_rows = rem;
        tiles = (rows - rem) + 2 * rem;
      }
    }
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((tiles < units ? tiles : units) * (CTA2 ? 2 : 1));
  cfg.blockDim = dim3(kGemmThreads);
  cfg.dynamicSmemBytes = SM::kBytes;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CTA2 ? 2 : 1;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, gp));
  return SCE_OK;
}

// Dispatch a K-major-A GEMM on (output width -> BN, K block, single CTA or CTA pair). Stage counts fill the
// 192 KB operand ring: single 256x{64,32} -> 2,4; 128x{64,32} -> 3,6; pair 256x{64,32} -> 3,6; 128x{64,32} -> 4,8.
// f16f8: K block 64 everywhere, a stage is one 16-bit plane of A and of B (or their four 8-bit planes): pair
// 256-wide -> 6 stages of 32 KB, single 256-wide -> 4 of 48 KB, single 128-wide -> 6 of 32 KB; narrow outputs
// never run on pairs (see build_maps).
template <class Epi, bool B_MN, bool SPLIT, int ARITH, class... Args>
static int launch_k(bool wide, int bk, bool pair, Args&&... a) {
  if constexpr (ARITH == kArithF16F8) {
    // epilogues that stage two chunks per bulk store take 8 KB per epilogue warp: one ring stage less
    constexpr int big = Epi::kWarpStageBytes > 4096 ? 1 : 0;
    if (wide)
      return pair ? launch_gemm_t<Epi, 256, kBkF8, false, B_MN, 6 - big, false, true, kArithF16F8>(a...)
                  : launch_gemm_t<Epi, 256, kBkF8, false, B_MN, 4 - big, false, false, kArithF16F8>(a...);
    return launch_gemm_t<Epi, 128, kBkF8, false, B_MN, 6 - big, false, false, kArithF16F8>(a...);
  } else {
  if (wide) {
    if (bk == 32)
      return pair ? launch_gemm_t<Epi, 256, 32, false, B_MN, 6, SPLIT, true>(a...)
                  : launch_gemm_t<Epi, 256, 32, false, B_MN, 4, SPLIT, false>(a...);
    return pair ? launch_gemm_t<Epi, 256, 64, false, B_MN, 3, SPLIT, true>(a...)
                : launch_gemm_t<Epi, 256, 64, false, B_MN, 2, SPLIT, false>(a...);
  }
  if (bk == 32)
    return pair ? launch_gemm_t<Epi, 128, 32, false, B_MN, 8, SPLIT, true>(a...)
                : launch_gemm_t<Epi, 128, 32, false, B_MN, 6, SPLIT, false>(a...);
  return pair ? launch_gemm_t<Epi, 128, 64, false, B_MN, 4, SPLIT, true>(a...)
              : launch_gemm_t<Epi, 128, 64, false, B_MN, 3, SPLIT, false>(a...);
  }
}

// ------------------------------------------------------------------------------------------------
// helpers shared by step / forward / grads
// ------------------------------------------------------------------------------------------------
static AdamHyper hyper_for(const sce_plan* p, long long t) {
  AdamHyper h;
  h.lr = p->d.lr;
  h.b1 = p->d.beta1;
  h.b2 = p->d.beta2;
  h.eps = p->d.eps;
  h.eps_root = p->d.eps_root;
  const double tt = p->d.adam_count_mode == SCE_ADAM_FROZEN_T1 ? 1.0 : (double)t;
  h.bc1 = (float)(1.0 - pow((double)h.b1, tt));
  h.bc2 = (float)(1.0 - pow((double)h.b2, tt));
  return h;
}

template <int MODE, int ARITH>
static int launch_dict_rows_t(float* e, const float* dw, float* m, float* v, void* hi, void* lo, void* x8,
                              float* grad_out, long long rows, int d, int normalize, float floor, AdamHyper h,
                              const uint32_t* health, float* w_f32, cudaStream_t st) {
  const int nv = (d + 511) / 512;
  if (nv == 1)
    dict_rows_kernel<1, MODE, ARITH><<<(unsigned)rows, 128, 0, st>>>(e, dw, m, v, hi, lo, x8, grad_out, d, normalize, floor, h, health, w_f32);
  else if (nv == 2)
    dict_rows_kernel<2, MODE, ARITH><<<(unsigned)rows, 128, 0, st>>>(e, dw, m, v, hi, lo, x8, grad_out, d, normalize, floor, h, health, w_f32);
  else if (nv <= 4)
    dict_rows_kernel<4, MODE, ARITH><<<(unsigned)rows, 128, 0, st>>>(e, dw, m, v, hi, lo, x8, grad_out, d, normalize, floor, h, health, w_f32);
  else if (nv <= 8)    // d <= 4096 (Pythia-6.9b residual width)
    dict_rows_kernel<8, MODE, ARITH><<<(unsigned)rows, 128, 0, st>>>(e, dw, m, v, hi, lo, x8, grad_out, d, normalize, floor, h, health, w_f32);
  else                 // d <= 8192
    dict_rows_kernel<16, MODE, ARITH><<<(unsigned)rows, 128, 0, st>>>(e, dw, m, v, hi, lo, x8, grad_out, d, normalize, floor, h, health, w_f32);
  CUDA_TRY(cudaGetLastError());
  return SCE_OK;
}
// `which`: 0 = the encoder's operand planes, 1 = the decoder's
template <int MODE>
static int launch_dict_rows(const sce_plan* p, int which, float* e, const float* dw, float* m, float* v, float* grad_out,
                            long long rows, int d, int normalize, float floor, AdamHyper h, cudaStream_t st) {
  void* hi = which ? (void*)p->wdec_hi : (void*)p->wenc_hi;
  void* lo = which ? (void*)p->wdec_lo : (void*)p->wenc_lo;
  void* x8 = which ? (void*)p->wdec_x8 : (void*)p->wenc_x8;
  if (MODE == MODE_GRAD) hi = lo = x8 = nullptr;
  float* wf = (MODE != MODE_GRAD && p->topk_sparse) ? p->wn_f32 : nullptr;   // (top-k plans have one dictionary)
  return p->arith == kArithF16F8
             ? launch_dict_rows_t<MODE, kArithF16F8>(e, dw, m, v, hi, lo, x8, grad_out, rows, d, normalize, floor, h, p->res_flags, wf, st)
             : launch_dict_rows_t<MODE, kArithBf16x3>(e, dw, m, v, hi, lo, x8, grad_out, rows, d, normalize, floor, h, p->res_flags, wf, st);
}

// f16f8 runs the backward pass on the residual r instead of g = 2r/(B d) (EpiDecodeT): weight- and bias-gradient
// outputs are multiplied by 2/(B d) on the way out, the sparsity term enters dcode as alpha d / 2.
static float grad_out_scale(const sce_plan* p, int B) {
  return p->arith == kArithF16F8 ? 2.0f / ((float)B * (float)p->d.d) : 1.0f;
}

__global__ void l1_over_b_kernel(const float* __restrict__ alpha, float* __restrict__ out, int M, float invB) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < M) out[i] = alpha ? alpha[i] * invB : 0.f;
}

// forward (+ optional backward GEMMs). Leaves dW in p->dw_enc / p->dw_dec when `backward`.
template <int AR>
static int run_pipeline_t(sce_plan* p, const float* x, int B, float* x_hat, bool backward, float* out_losses,
                          float* out_nnz, cudaStream_t st) {
  using EpiEnc = EpiEncodeT<AR>;
  using EpiDec = EpiDecodeT<AR>;
  using EpiDco = EpiDcodeT<AR>;
  constexpr bool f8 = AR == kArithF16F8;
  const sce_desc& d = p->d;
  if (B < 1 || B > d.batch_max) return fail(SCE_ERR_INVALID, "B = %d outside [1, batch_max = %d]", B, d.batch_max);
  if (!x) return fail(SCE_ERR_INVALID, "x is NULL");
  BatchMaps* maps = nullptr;
  int rc = build_maps(p, B, &maps);
  if (rc) return rc;
  int launches = 0;
  const int M = d.n_models, n = d.n, dd = d.d;
  const long long Bm = d.batch_max;
  const int one[2] = {1, 1};
  const int xb[2] = {d.x_per_model ? 1 : 0, 1};
  const int tiles_mB = (B + kBM - 1) / kBM;

  prof_mark(p, SCE_PHASE_SPLIT, st);
  // the f16f8 kernels run narrow outputs on single CTAs (build_maps)
  auto pair_ok = [&](int flag, int rows, int out_cols) { return use_pair(flag, rows) && !(f8 && out_cols <= 128); };
  if (d.centering) {
    // ---- centring (sae_ensemble.py:126-128): (x - trans[m]) -> planes, GEMM with rot[m] (all split passes), * scale[m]
    // -> the per-model fp32 batch every kernel below reads as `x`
    const long long n4 = (long long)B * dd / 4;
    const int blocks = (int)((n4 + 255) / 256 < 1024 ? (n4 + 255) / 256 : 1024);
    center_split_kernel<AR><<<dim3(blocks, M), 256, 0, st>>>(
        x, d.centering == 2 ? (long long)B * dd : 0, p->b.center_trans, p->x_hi, p->x_lo, p->x_x8, Bm * dd, B, dd);
    CUDA_TRY(cudaGetLastError());
    EpiCenter::Params cp;
    cp.out = p->x_centered;
    cp.model_stride = (long long)B * dd;
    cp.ld = dd;
    cp.col_scale = p->b.center_scale;
    rc = launch_k<EpiCenter, false, false, AR>(dd > 128, p->bk_encode, pair_ok(p->pair_encode, B, dd), p, maps->center, 1, one, one,
                                              dd, 3, B, dd, cp, st);
    if (rc) return rc;
    launches += 2;
    x = p->x_centered;
  }
  // ---- x -> (hi, lo): per model slabs are batch_max apart in the workspace
  if constexpr (f8) CUDA_TRY(cudaMemsetAsync(p->res_flags, 0, sizeof(uint32_t), st));
  for (int m = 0; m < p->xm; ++m) {
    const long long n4 = (long long)B * dd / 4;
    const int blocks = (int)((n4 + 255) / 256 < 2048 ? (n4 + 255) / 256 : 2048);
    // (bf16x3: the lo plane is 2 B / element; f16f8: lo and x8 are 1 B / element)
    split_rows_kernel<AR><<<blocks, 256, 0, st>>>(
        x + (long long)m * B * dd, p->x_hi + m * Bm * dd,
        f8 ? (void*)(reinterpret_cast<uint8_t*>(p->x_lo) + m * Bm * dd) : (void*)(p->x_lo + m * Bm * dd),
        f8 ? (void*)(p->x_x8 + m * Bm * dd) : nullptr, n4, f8 ? p->res_flags : nullptr);
    ++launches;
  }
  CUDA_TRY(cudaGetLastError());
  // alpha / B, or (f16f8, backward on r = g B d / 2) alpha d / 2
  l1_over_b_kernel<<<(M + 127) / 128, 128, 0, st>>>(p->b.l1_alpha, p->l1_over_b, M, f8 ? 0.5f * (float)dd : 1.0f / (float)B);
  ++launches;
  // the batch's residual-plane flag, for the GEMMs that read x as their A (encode) or B (weight gradient, set 0) operand
  ResFlags x_is_a, x_is_b;
  if constexpr (f8) {
    x_is_a.a[0] = p->res_flags;
    x_is_b.b[0] = p->res_flags;
  }
  ActMask act;
  act.pos = p->act_pos;
  act.zero = p->act_zero;
  act.n_chunks = (n + 31) / 32;
  act.batch_max = d.batch_max;
  if (d.variant == SCE_TOPK) act.zero = nullptr;   // relu semantics: no gradient at exactly 0
  // ---- encode
  prof_mark(p, SCE_PHASE_ENCODE, st);
  int n_enc_parts;
  TopkLists tk = {nullptr, nullptr, nullptr, 0, 0};
  if (d.variant != SCE_TOPK) {
    typename EpiEnc::Params ep;
    ep.out_hi = maps->st_c_hi;
    ep.out_lo = maps->st_c_lo;
    ep.out_x8 = maps->st_c_x8;
    ep.bias = p->b.encoder_bias;
    ep.mask = p->b.coef_mask;
    ep.part = p->part_enc;
    ep.tiles_m = tiles_mB;
    ep.flag_zero = 1;
    ep.act = act;
    ep.tiles_n = n > 128 ? (n + 255) / 256 : 1;
    rc = launch_k<EpiEnc, false, false, AR>(n > 128, p->bk_encode, pair_ok(p->pair_encode, B, n), p, maps->encode, 1, xb, one,
                                            dd, d.fwd_passes, B, n, ep, st, x_is_a);
    if (rc) return rc;
    ++launches;
    n_enc_parts = tiles_mB * 8 * ep.tiles_n;
  } else {
    // scores -> fp32, then per-row selection (code planes, activity mask, k-sparse lists)
    EpiScoresTma::Params sp;
    sp.out = maps->st_scores;
    if (p->topk_cmax) {
      sp.cmax = p->tk_cmax;
      sp.n_chunks = act.n_chunks;
      sp.cmax_model_stride = (long long)Bm * act.n_chunks;
    }
    rc = launch_k<EpiScoresTma, false, false, AR>(n > 128, p->bk_encode, pair_ok(p->pair_encode, B, n), p, maps->encode, 1, xb,
                                                 one, dd, d.fwd_passes, B, n, sp, st, x_is_a);
    if (rc) return rc;
    ++launches;
    static bool cfg[64] = {};
    if (p->device < 0 || p->device >= 64 || !cfg[p->device]) {
      CUDA_TRY(cudaFuncSetAttribute(topk_sparse_kernel<AR>, cudaFuncAttributeMaxDynamicSharedMemorySize, 112 * 1024));
      if (p->device >= 0 && p->device < 64) cfg[p->device] = true;
    }
    tk.col = p->tk_col;
    tk.val = p->tk_val;
    tk.cnt = p->tk_cnt;
    tk.kmax = p->tk_kmax;
    tk.batch_max = d.batch_max;
    // one block per (row, model); scores / codes of model m start at m * batch_max * n
    topk_select2_kernel<AR><<<dim3(B, M), 256, 0, st>>>(
        p->scores, p->b.sparsity, p->c_hi, p->c_lo, p->c_x8, p->topk_sparse ? (void*)p->dz_hi : nullptr, p->dz_lo, p->dz_x8,
        act, tk, p->part_enc, B, n, Bm * n, p->topk_cmax ? p->tk_cmax : nullptr);
    ++launches;
    CUDA_TRY(cudaGetLastError());
    n_enc_parts = B;
  }

  const bool sparse = d.variant == SCE_TOPK && p->topk_sparse;
  int n_dec_parts;
  prof_mark(p, SCE_PHASE_DECODE, st);
  if (sparse) {
    // ---- k-sparse decode + residual + loss partial + g planes + the code gradient at the selected entries
    const float gscale = f8 ? 1.0f : 2.0f / ((float)B * (float)dd);
    // one launch per k class (sce_prepare sorted the models): a block's shared memory goes with ITS models' k, so the
    // k = 16 and k = 32 models of a mixed ensemble run at 5 and 3 blocks per SM instead of the 2 that k_max = 64 allows
    for (int g = 0; g < p->tk_groups; ++g) {
      const int cnt = p->tk_group_off[g + 1] - p->tk_group_off[g];
      if (cnt == 0) continue;
      topk_sparse_kernel<AR><<<dim3(B, cnt, p->tk_slices), 256, topk_sparse_smem(d, p->tk_group_krows[g], p->tk_slices), st>>>(
          tk, p->b.sparsity, p->wn_f32, x, d.x_per_model ? (long long)B * dd : 0, p->g_hi, p->g_lo, p->g_x8, x_hat, p->part_dec,
          backward ? p->tk_dots : nullptr, B, n, dd, gscale, p->tk_models + p->tk_group_off[g], p->tk_group_krows[g]);
      ++launches;
    }
    CUDA_TRY(cudaGetLastError());
    n_dec_parts = p->tk_slices * B;
  } else {
  // ---- decode (+ residual, loss partial, g)
  typename EpiDec::Params dp;
  dp.x = x;
  dp.x_model_stride = d.x_per_model ? (long long)B * dd : 0;
  dp.g_hi = reinterpret_cast<uint16_t*>(p->g_hi);
  dp.g_lo = reinterpret_cast<uint8_t*>(p->g_lo);
  dp.g_x8 = p->g_x8;
  dp.x_hat = x_hat;
  dp.part = p->part_dec;
  dp.g_model_stride = Bm * dd;
  dp.xhat_model_stride = (long long)B * dd;
  dp.ld = dd;
  dp.tiles_m = tiles_mB;
  dp.gscale = f8 ? 1.0f : 2.0f / ((float)B * (float)dd);
  dp.tiles_n = dd > 128 ? (dd + 255) / 256 : 1;
  if (f8 && p->dec_nsub2 && dd % 512 == 0 && pair_ok(p->pair_decode, B, dd)) {
    // experiment (SCE_TUNE_DEC_NSUB2=1): 256 x 512 tiles — the code tile (A) read once for both column halves, kept in the
    // collector; the accumulators fill all of tensor memory, so the epilogue no longer overlaps the next main loop
    if constexpr (f8)
      rc = launch_gemm_t<EpiDec, 256, kBkF8, false, true, 4, false, true, kArithF16F8, 2>(p, maps->decode, 1, one, one, n, d.fwd_passes,
                                                                                      B, dd, dp, st);
  } else if (p->split_decode && !f8)
    rc = launch_k<EpiDec, true, true, AR>(dd > 128, p->bk_decode, pair_ok(p->pair_decode, B, dd), p, maps->decode, 1, one, one,
                                          n, d.fwd_passes, B, dd, dp, st);
  else
    rc = launch_k<EpiDec, true, false, AR>(dd > 128, p->bk_decode, pair_ok(p->pair_decode, B, dd), p, maps->decode, 1, one, one,
                                           n, d.fwd_passes, B, dd, dp, st);
  if (rc) return rc;
  ++launches;
  n_dec_parts = tiles_mB * 8 * dp.tiles_n;
  }

  // ---- losses
  prof_mark(p, SCE_PHASE_LOSSES, st);
  if (p->b.encoder_bias && p->b.bias_decay) {
    bias_norm_kernel<<<M, 256, 0, st>>>(p->b.encoder_bias, n, p->bnorm);
    ++launches;
  }
  finalize_kernel<<<M, 256, 0, st>>>(p->part_enc, n_enc_parts, p->part_dec, n_dec_parts, p->b.l1_alpha,
                                     p->b.encoder_bias ? p->b.bias_decay : nullptr, p->bnorm, B, dd, out_losses, out_nnz,
                                     p->res_flags);
  ++launches;
  CUDA_TRY(cudaGetLastError());

  prof_mark(p, SCE_PHASE_DCODE, st);
  if (backward) {
    if (sparse) {
      // ---- code gradient planes: zero the rows, scatter the k entries
      topk_dz_scatter_kernel<AR><<<dim3(B, M), 64, 0, st>>>(tk, p->tk_dots, p->tk_slices, p->dz_hi, p->dz_lo, p->dz_x8, n);
      ++launches;
      CUDA_TRY(cudaGetLastError());
    } else {
    // ---- dcode
    typename EpiDco::Params zp;
    zp.out_hi = maps->st_dz_hi;
    zp.out_lo = maps->st_dz_lo;
    zp.out_x8 = maps->st_dz_x8;
    zp.act = act;
    zp.l1_over_b = p->l1_over_b;
    zp.db_part = p->b.encoder_bias ? p->db_part : nullptr;
    zp.tiles_m = tiles_mB;
    zp.planes = p->dw_passes >= 3 ? 3 : 0;
    // the only reader of dz's value plane is the dz^T x term of the weight gradient, against x's residual plane
    // (per-model batches carry one flag for all of them, so the same test holds)
    zp.x_res_flag = f8 ? p->res_flags : nullptr;
    rc = launch_k<EpiDco, false, false, AR>(n > 128, p->bk_dcode, pair_ok(p->pair_dcode, B, n), p, maps->dcode, 1, one, one, dd,
                                            p->dcode_passes, B, n, zp, st);
    if (rc) return rc;
    ++launches;
    }

    // ---- weight gradients
    prof_mark(p, SCE_PHASE_DW, st);
    auto dw = [&](const GemmMaps& gm, int nsets, const int* ab, const int* bb, float* out, const ResFlags& rf) -> int {
      EpiStoreF32::Params sp;
      sp.out = out;
      sp.model_stride = (long long)n * dd;
      sp.ld = dd;
      sp.scale = grad_out_scale(p, B);
      const bool pair = pair_ok(p->pair_dw, n, dd);
      if constexpr (f8) {
        // d > 256: both 256-column halves of a dictionary row block from one A (dz / c) tile per K block (NSUB = 2)
        if (dd % 512 == 0 && pair && p->dw_nsub2)
          return launch_gemm_t<EpiStoreF32, 256, kBkF8, true, true, 4, false, true, kArithF16F8, 2>(p, gm, nsets, ab, bb, B, p->dw_passes, n, dd, sp, st, rf);
        if (dd > 128)
          return pair ? launch_gemm_t<EpiStoreF32, 256, kBkF8, true, true, 6, false, true, kArithF16F8>(p, gm, nsets, ab, bb, B, p->dw_passes, n, dd, sp, st, rf)
                      : launch_gemm_t<EpiStoreF32, 256, kBkF8, true, true, 4, false, false, kArithF16F8>(p, gm, nsets, ab, bb, B, p->dw_passes, n, dd, sp, st, rf);
        return launch_gemm_t<EpiStoreF32, 128, kBkF8, true, true, 6, false, false, kArithF16F8>(p, gm, nsets, ab, bb, B, p->dw_passes, n, dd, sp, st, rf);
      }
      if (dd > 128)
        return pair ? launch_gemm_t<EpiStoreF32, 256, kBkDw, true, true, 6, true, true>(p, gm, nsets, ab, bb, B, p->dw_passes, n, dd, sp, st)
                    : launch_gemm_t<EpiStoreF32, 256, kBkDw, true, true, 4, true, false>(p, gm, nsets, ab, bb, B, p->dw_passes, n, dd, sp, st);
      return pair ? launch_gemm_t<EpiStoreF32, 128, kBkDw, true, true, 8, true, true>(p, gm, nsets, ab, bb, B, p->dw_passes, n, dd, sp, st)
                  : launch_gemm_t<EpiStoreF32, 128, kBkDw, true, true, 6, true, false>(p, gm, nsets, ab, bb, B, p->dw_passes, n, dd, sp, st);
    };
    if (d.variant == SCE_UNTIED) {
      rc = dw(maps->dw_enc, 1, one, xb, p->dw_enc, x_is_b);
      if (rc) return rc;
      rc = dw(maps->dw_dec, 1, one, one, p->dw_dec, ResFlags());
      if (rc) return rc;
      launches += 2;
    } else {
      const int bb[2] = {xb[0], 1};
      rc = dw(maps->dw_enc, 2, one, bb, p->dw_enc, x_is_b);
      if (rc) return rc;
      ++launches;
    }
  }
  prof_mark(p, SCE_PHASE_ADAM, st);
  p->last_launches = launches;
  return SCE_OK;
}

static int run_pipeline(sce_plan* p, const float* x, int B, float* x_hat, bool backward, float* out_losses,
                        float* out_nnz, cudaStream_t st) {
  return p->arith == kArithF16F8 ? run_pipeline_t<kArithF16F8>(p, x, B, x_hat, backward, out_losses, out_nnz, st)
                                 : run_pipeline_t<kArithBf16x3>(p, x, B, x_hat, backward, out_losses, out_nnz, st);
}

// ------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------
extern "C" {

int sce_version(void) { return SCE_VERSION; }
const char* sce_last_error(void) { return g_err; }

size_t sce_workspace_bytes(const sce_desc* desc) {
  if (validate(desc)) return 0;
  return carve(nullptr, *desc, nullptr);
}

int sce_plan_create(const sce_desc* desc, const sce_buffers* buffers, sce_plan** out_plan) {
  if (!out_plan) return fail(SCE_ERR_INVALID, "out_plan is NULL");
  *out_plan = nullptr;
  int rc = validate(desc);
  if (rc) return rc;
  if (!buffers) return fail(SCE_ERR_INVALID, "buffers is NULL");
  const sce_buffers& b = *buffers;
  if (!b.encoder || !b.encoder_m || !b.encoder_v) return fail(SCE_ERR_INVALID, "encoder / encoder_m / encoder_v are required");
  if (desc->variant == SCE_UNTIED && (!b.decoder || !b.decoder_m || !b.decoder_v))
    return fail(SCE_ERR_INVALID, "untied variant needs decoder / decoder_m / decoder_v");
  if (desc->variant != SCE_TOPK && (!b.encoder_bias || !b.bias_m || !b.bias_v))
    return fail(SCE_ERR_INVALID, "encoder_bias / bias_m / bias_v are required for SAE variants");
  if (desc->variant == SCE_TOPK && !b.sparsity) return fail(SCE_ERR_INVALID, "top-k variant needs the sparsity buffer");
  const size_t need = carve(nullptr, *desc, nullptr);
  if (!b.workspace || b.workspace_bytes < need)
    return fail(SCE_ERR_WORKSPACE, "workspace too small: have %zu bytes, need %zu", b.workspace_bytes, need);
  if (reinterpret_cast<uintptr_t>(b.workspace) % 1024)
    return fail(SCE_ERR_WORKSPACE, "workspace must be 1024-byte aligned");
  int dev = 0, major = 0, sms = 0;
  CUDA_TRY(cudaGetDevice(&dev));
  CUDA_TRY(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  if (major != 10) return fail(SCE_ERR_NO_DEVICE, "libsce needs an sm_100 device (found compute capability %d.x)", major);
  if (!get_encode_fn()) return fail(SCE_ERR_NO_DEVICE, "cuTensorMapEncodeTiled driver entry point not available");
  sce_plan* p = new (std::nothrow) sce_plan;
  if (!p) return fail(SCE_ERR_INVALID, "out of host memory");
  memset(p, 0, sizeof(*p));
  p->d = *desc;
  p->b = b;
  p->sms = sms;
  p->device = dev;
  p->xm = desc->x_per_model ? desc->n_models : 1;
  p->arith = resolve_arith(*desc);
  // CTA pairs by default for all four GEMMs (same-box A/B in profiles/r01g_pair_tuning.txt: -10 % encode,
  // -9 % decode, -3 % dcode, -21 % weight gradient on that box; env SCE_TUNE_PAIR_* = 0 switches one back)
  p->pair_encode = tune_flag("SCE_TUNE_PAIR_ENCODE", 1);
  p->pair_decode = tune_flag("SCE_TUNE_PAIR_DECODE", 1);
  p->pair_dcode = tune_flag("SCE_TUNE_PAIR_DCODE", 1);
  p->pair_dw = tune_flag("SCE_TUNE_PAIR_DW", 1);
  // The truncation bias of a single accumulation chain grows with the reduction length (about 3.7e-9 * n on x_hat,
  // up to ~3.6x that on the loss): harmless at n <= 4096 (1.5e-5 / 3e-5 measured), over the 1e-4 bar near
  // n = 16384-32768. Splitting costs the decode GEMM its accumulator double-buffering (1.14 -> 1.29 ms at config 2,
  // profiles/r01i_split_decode_tuning.txt), so it is switched on where it is needed.
  p->split_decode = tune_flag("SCE_TUNE_SPLIT_DECODE", desc->n > 4096 ? 1 : 0);
  p->dcode_passes = desc->bwd_passes;
  p->dw_passes = desc->bwd_passes;
  if (const char* v = getenv("SCE_TUNE_DCODE_PASSES")) p->dcode_passes = atoi(v) == 1 ? 1 : 3;
  if (const char* v = getenv("SCE_TUNE_DW_PASSES")) p->dw_passes = atoi(v) == 1 ? 1 : 3;
  {
    // ~30 M B n d tensor FLOPs are issued per step; below ~3e11 (a fifth of a millisecond) launches dominate
    const double issued = 30.0 * desc->n_models * (double)desc->batch_max * desc->n * desc->d;
    p->use_graph = tune_flag("SCE_GRAPH", issued < 3e11 ? 1 : 0);
  }
  // 256 x 512 weight-gradient tiles (one A tile for both column halves): DRAM traffic of the launch 5.69 -> 4.25 GB
  // at config 2, device time unchanged within the run-to-run noise (1.51 / 1.50 / 1.57 ms against 1.51 / 1.50 ms: the
  // kernel is bound by the power-limited tensor rate either way) — off by default, kept as a knob
  p->dw_nsub2 = tune_flag("SCE_TUNE_DW_NSUB2", 1);
  p->dw_collector = tune_flag("SCE_TUNE_DW_COLL", 1);
  p->dec_nsub2 = tune_flag("SCE_TUNE_DEC_NSUB2", 0);
  p->bk_encode = tune_bk("SCE_TUNE_BK_ENCODE", 64);
  p->bk_decode = tune_bk("SCE_TUNE_BK_DECODE", 32);
  p->bk_dcode = tune_bk("SCE_TUNE_BK_DCODE", 64);
  {
    // k-sparse decode / dcode of the top-k variant: lists known (topk_k_max), bulk-copy alignment of the dictionary
    // half rows (16 bytes in every plane), shared memory of the gather kernel
    const size_t kmax = topk_kmax(*desc);
    p->tk_slices = kmax ? topk_slices(*desc, kmax) : 0;
    if (const char* v = getenv("SCE_TOPK_SLICES")) {
      const int sl = atoi(v);
      if (kmax && (sl == 2 || sl == 4 || sl == 8) && desc->d % (4 * sl) == 0 && desc->d / sl <= 512 &&
          topk_sparse_smem(*desc, kmax, sl) <= 112 * 1024)
        p->tk_slices = sl;
    }
    // Worth it where the dictionary is large against k: the dense decode + dcode GEMMs cost ~ n per row, the gather
    // kernel ~ k (it is bound by the latency chain of a block, not by bytes). Measured on B200, d = 768, 12 models,
    // k in {16, 32, 64}, one launch per k class (tools/run_r02w.sh): n = 6144 dense 1.40 + 1.50 ms / sparse 2.56 + 0.31 ms —
    // equal as kernels, but the step with the gather path is 4 % shorter (7.83 against 8.17 ms: the GPU runs these steps
    // at its power cap and the gather kernel leaves the tensor pipes idle); n = 12288 dense 5.8 ms / sparse 2.9 ms;
    // n = 3072: config 3 with every group on the gather path 22.26 ms against an estimated 22.15 ms with this rule.
    // SCE_TOPK_SPARSE = 1 / 0 forces it on / off.
    const int heuristic = (long long)desc->n >= 96ll * (long long)(kmax ? kmax : 1);
    p->topk_sparse = desc->variant == SCE_TOPK && kmax > 0 && p->tk_slices > 0 && tune_flag("SCE_TOPK_SPARSE", heuristic);
    // selection from the per-chunk maxima the scores epilogue writes (profiles/r02p_*); 0 = read every row twice as before
    p->topk_cmax = desc->variant == SCE_TOPK && tune_flag("SCE_TOPK_CMAX", 1);
  }
  p->maps = new std::map<int, BatchMaps*>();
  carve(p, *desc, static_cast<uint8_t*>(b.workspace));
  *out_plan = p;
  return SCE_OK;
}

int sce_plan_destroy(sce_plan* plan) {
  if (!plan) return SCE_OK;
  for (auto& kv : *plan->maps) {
    if (kv.second->graph) cudaGraphExecDestroy(kv.second->graph);
    delete kv.second;
  }
  delete plan->maps;
  if (plan->cap_stream) cudaStreamDestroy(plan->cap_stream);
  if (plan->prof_ev) {
    for (int i = 0; i < kProfMaxSteps * (SCE_PHASE_COUNT + 1); ++i) cudaEventDestroy(plan->prof_ev[i]);
    free(plan->prof_ev);
  }
  delete plan;
  return SCE_OK;
}

int sce_prepare(sce_plan* p, void* stream) {
  if (!p) return fail(SCE_ERR_INVALID, "plan is NULL");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CUDA_TRY(cudaMemsetAsync(p->res_flags, 0, kFlagWords * sizeof(uint32_t), st));   // residual flag, input range monitor, health
  const sce_desc& d = p->d;
  const long long rows = (long long)d.n_models * d.n;
  std::vector<long long> ks;
  if (d.variant == SCE_TOPK) {
    // the selection kernel takes k from buffers.sparsity as it is: k < 1 leaves its bound unset, and a plan with lists
    // records at most its capacity of the k entries it scatters, so the next call would not clear the others
    ks.resize(d.n_models);
    CUDA_TRY(cudaMemcpyAsync(ks.data(), p->b.sparsity, ks.size() * sizeof(long long), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    for (int m = 0; m < d.n_models; ++m) {
      if (ks[m] < 1 || ks[m] > d.n)
        return fail(SCE_ERR_INVALID, "model %d: sparsity k = %lld outside [1, n = %d]", m, ks[m], d.n);
      if (p->tk_kmax && ks[m] > d.topk_k_max)
        return fail(SCE_ERR_INVALID, "model %d: sparsity k = %lld above the plan's topk_k_max = %d (create a new plan)", m,
                    ks[m], d.topk_k_max);
    }
  }
  if (d.variant == SCE_TOPK && p->tk_kmax) {
    // the top-k selection keeps the code planes (and, in k-sparse plans, the code-gradient planes) all-zero except for
    // the entries its lists record: start them zeroed, with empty lists
    const size_t el = (size_t)d.n_models * d.batch_max * d.n;
    const bool f8 = p->arith == kArithF16F8;
    CUDA_TRY(cudaMemsetAsync(p->c_hi, 0, el * 2, st));
    CUDA_TRY(cudaMemsetAsync(p->c_lo, 0, el * (f8 ? 1 : 2), st));
    if (f8) CUDA_TRY(cudaMemsetAsync(p->c_x8, 0, el, st));
    CUDA_TRY(cudaMemsetAsync(p->dz_hi, 0, el * 4, st));   // (the code-gradient planes are one contiguous block, 4 B / element)
    CUDA_TRY(cudaMemsetAsync(p->act_pos, 0, (size_t)d.n_models * ((d.n + 31) / 32) * d.batch_max * sizeof(uint32_t), st));
    CUDA_TRY(cudaMemsetAsync(p->tk_cnt, 0, (size_t)d.n_models * d.batch_max * sizeof(int), st));
    // k classes for the gather kernel: rows of shared memory in {16, 32, 64} and the list capacity, each capped at it
    const int caps[4] = {16, 32, 64, p->tk_kmax};
    std::vector<int> order;
    p->tk_groups = 0;
    p->tk_group_off[0] = 0;
    int lo = 0;
    for (int g = 0; g < 4; ++g) {
      const int cap = caps[g] < p->tk_kmax ? caps[g] : p->tk_kmax;
      if (g > 0 && cap <= lo) continue;
      for (int m = 0; m < d.n_models; ++m) {
        if (ks[m] > lo && ks[m] <= cap) order.push_back(m);   // (1 <= k <= topk_k_max <= tk_kmax: checked above)
      }
      p->tk_group_krows[p->tk_groups] = cap;
      p->tk_group_off[++p->tk_groups] = (int)order.size();
      lo = cap;
      if (cap == p->tk_kmax) break;
    }
    if ((int)order.size() != d.n_models) return fail(SCE_ERR_INVALID, "top-k classes: %d of %d models placed", (int)order.size(), d.n_models);
    CUDA_TRY(cudaMemcpyAsync(p->tk_models, order.data(), order.size() * sizeof(int), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaStreamSynchronize(st));   // (`order` is a local)
  }
  if (d.centering) {
    if (!p->b.center_trans || !p->b.center_rot || !p->b.center_scale)
      return fail(SCE_ERR_INVALID, "centering needs the center_trans / center_rot / center_scale buffers");
    const long long n4 = (long long)d.n_models * d.d * d.d / 4;
    const int blocks = (int)((n4 + 255) / 256 < 2048 ? (n4 + 255) / 256 : 2048);
    if (p->arith == kArithF16F8)
      split_rows_kernel<kArithF16F8><<<blocks, 256, 0, st>>>(p->b.center_rot, p->rot_hi, p->rot_lo, p->rot_x8, n4, nullptr);
    else
      split_rows_kernel<kArithBf16x3><<<blocks, 256, 0, st>>>(p->b.center_rot, p->rot_hi, p->rot_lo, nullptr, n4, nullptr);
    CUDA_TRY(cudaGetLastError());
  }
  AdamHyper h = hyper_for(p, 1);
  int rc;
  if (d.variant == SCE_UNTIED) {
    rc = launch_dict_rows<MODE_PREPARE>(p, 0, p->b.encoder, nullptr, nullptr, nullptr, nullptr, rows, d.d, 0, 0.f, h, st);
    if (rc) return rc;
    rc = launch_dict_rows<MODE_PREPARE>(p, 1, p->b.decoder, nullptr, nullptr, nullptr, nullptr, rows, d.d, 1, d.norm_floor, h, st);
  } else {
    rc = launch_dict_rows<MODE_PREPARE>(p, 0, p->b.encoder, nullptr, nullptr, nullptr, nullptr, rows, d.d, 1, d.norm_floor, h, st);
  }
  return rc;
}

int sce_forward(sce_plan* p, const float* x, int B, float* x_hat, float* out_losses, float* out_nnz, void* stream) {
  if (!p) return fail(SCE_ERR_INVALID, "plan is NULL");
  return run_pipeline(p, x, B, x_hat, false, out_losses, out_nnz, static_cast<cudaStream_t>(stream));
}

// models' worth of rows in the caller's batch: 1 when it is shared ([B,d]; also with centering = 1), else M
static int input_models(const sce_plan* p) { return p->d.centering == 1 ? 1 : p->xm; }

// every launch of one optimisation step, in order, on `st` (also what gets captured into a CUDA graph)
static int step_launches(sce_plan* p, const float* x, int B, float* out_losses, float* out_nnz, long long t,
                         cudaStream_t st) {
  int rc = run_pipeline(p, x, B, nullptr, true, out_losses, out_nnz, st);
  if (rc) return rc;
  const sce_desc& d = p->d;
  const long long rows = (long long)d.n_models * d.n;
  const AdamHyper h = hyper_for(p, t);
  int launches = p->last_launches;
  if (d.variant == SCE_UNTIED) {
    rc = launch_dict_rows<MODE_ADAM>(p, 0, p->b.encoder, p->dw_enc, p->b.encoder_m, p->b.encoder_v, nullptr, rows, d.d, 0,
                                     0.f, h, st);
    if (rc) return rc;
    rc = launch_dict_rows<MODE_ADAM>(p, 1, p->b.decoder, p->dw_dec, p->b.decoder_m, p->b.decoder_v, nullptr, rows, d.d, 1,
                                     d.norm_floor, h, st);
    if (rc) return rc;
    launches += 2;
  } else {
    rc = launch_dict_rows<MODE_ADAM>(p, 0, p->b.encoder, p->dw_enc, p->b.encoder_m, p->b.encoder_v, nullptr, rows, d.d, 1,
                                     d.norm_floor, h, st);
    if (rc) return rc;
    ++launches;
  }
  if (p->b.encoder_bias) {
    const long long tot = (long long)d.n_models * d.n;
    const int n_part = ((B + kBM - 1) / kBM) * 4;
    bias_kernel<MODE_ADAM><<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(
        p->b.encoder_bias, p->b.bias_m, p->b.bias_v, p->db_part, n_part, d.n, d.n_models, p->b.bias_decay, p->bnorm,
        nullptr, h, grad_out_scale(p, B), p->res_flags);
    CUDA_TRY(cudaGetLastError());
    ++launches;
  }
  prof_mark(p, SCE_PHASE_COUNT, st);
  p->last_launches = launches;
  return SCE_OK;
}

// Launch-bound shapes (a step of ~10 kernels that each run a few microseconds, e.g. BASELINE config 1) replay the
// step as one CUDA graph: the batch is first copied into the plan's staging buffer so that every kernel argument is
// stable, the graph is captured on the second step at a given batch size (the first one runs eagerly and performs
// the one-off cudaFuncSetAttribute calls); the captured kernels write the plan's staging outputs, which are copied to
// the caller's buffers after the launch.
static bool graph_eligible(const sce_plan* p) {
  if (p->prof_on) return false;                                   // per-phase events are recorded eagerly
  if (p->d.adam_count_mode != SCE_ADAM_FROZEN_T1) return false;   // bias correction is a kernel argument that moves
  return p->use_graph != 0;
}

int sce_step(sce_plan* p, const float* x, int B, float* out_losses, float* out_nnz, void* stream) {
  if (!p) return fail(SCE_ERR_INVALID, "plan is NULL");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (B < 1 || B > p->d.batch_max) return fail(SCE_ERR_INVALID, "B = %d outside [1, batch_max = %d]", B, p->d.batch_max);
  if (!x) return fail(SCE_ERR_INVALID, "x is NULL");
  int rc;
  if (!graph_eligible(p)) {
    rc = step_launches(p, x, B, out_losses, out_nnz, p->step + 1, st);
  } else {
    BatchMaps* maps = nullptr;
    rc = build_maps(p, B, &maps);
    if (rc) return rc;
    const size_t bytes = (size_t)input_models(p) * B * p->d.d * sizeof(float);
    if (x != p->x_stage) CUDA_TRY(cudaMemcpyAsync(p->x_stage, x, bytes, cudaMemcpyDeviceToDevice, st));
    // the captured kernels write the plan's own staging outputs (stable addresses: callers may pass fresh tensors
    // every step, as the reference returns them); the results are copied out below
    float* const cap_losses = p->loss_stage;
    float* const cap_nnz = p->nnz_stage;
    if (maps->graph) {
      CUDA_TRY(cudaGraphLaunch(maps->graph, st));
      p->last_launches = maps->graph_launches;
      rc = SCE_OK;
    } else if (maps->eager_steps == 0) {
      maps->eager_steps = 1;
      rc = step_launches(p, p->x_stage, B, cap_losses, cap_nnz, 1, st);
    } else {
      // capture on a private stream (the caller's may be the legacy default stream, which cannot be captured);
      // capturing records the launches without running them, the instantiated graph is launched on `st`
      cudaGraph_t g = nullptr;
      if (!p->cap_stream) CUDA_TRY(cudaStreamCreateWithFlags(&p->cap_stream, cudaStreamNonBlocking));
      CUDA_TRY(cudaStreamBeginCapture(p->cap_stream, cudaStreamCaptureModeThreadLocal));
      rc = step_launches(p, p->x_stage, B, cap_losses, cap_nnz, 1, p->cap_stream);
      cudaError_t ce = cudaStreamEndCapture(p->cap_stream, &g);
      if (rc == SCE_OK && ce == cudaSuccess && g) {
        cudaGraphExec_t ge = nullptr;
        ce = cudaGraphInstantiate(&ge, g, 0);
        cudaGraphDestroy(g);
        if (ce != cudaSuccess) return fail(SCE_ERR_CUDA, "cudaGraphInstantiate failed: %s", cudaGetErrorString(ce));
        maps->graph = ge;
        maps->graph_launches = p->last_launches;
        CUDA_TRY(cudaGraphLaunch(maps->graph, st));
      } else {
        if (g) cudaGraphDestroy(g);
        cudaGetLastError();
        if (rc == SCE_OK) return fail(SCE_ERR_CUDA, "stream capture of the step failed: %s", cudaGetErrorString(ce));
      }
    }
    if (rc == SCE_OK && out_losses && out_losses != cap_losses)
      CUDA_TRY(cudaMemcpyAsync(out_losses, cap_losses, (size_t)p->d.n_models * SCE_LOSS_COLS * sizeof(float),
                               cudaMemcpyDeviceToDevice, st));
    if (rc == SCE_OK && out_nnz && out_nnz != cap_nnz)
      CUDA_TRY(cudaMemcpyAsync(out_nnz, cap_nnz, (size_t)p->d.n_models * sizeof(float), cudaMemcpyDeviceToDevice, st));
  }
  if (rc) return rc;
  p->step += 1;
  if (p->prof_on && p->prof_steps < kProfMaxSteps) p->prof_steps += 1;
  return SCE_OK;
}

int sce_grads(sce_plan* p, const float* x, int B, float* d_encoder, float* d_bias, float* d_decoder,
              float* out_losses, float* out_nnz, void* stream) {
  if (!p) return fail(SCE_ERR_INVALID, "plan is NULL");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int rc = run_pipeline(p, x, B, nullptr, true, out_losses, out_nnz, st);
  if (rc) return rc;
  const sce_desc& d = p->d;
  const long long rows = (long long)d.n_models * d.n;
  const AdamHyper h = hyper_for(p, 1);
  if (d.variant == SCE_UNTIED) {
    if (d_encoder) {
      rc = launch_dict_rows<MODE_GRAD>(p, 0, p->b.encoder, p->dw_enc, nullptr, nullptr, d_encoder, rows, d.d, 0, 0.f, h, st);
      if (rc) return rc;
    }
    if (d_decoder) {
      rc = launch_dict_rows<MODE_GRAD>(p, 1, p->b.decoder, p->dw_dec, nullptr, nullptr, d_decoder, rows, d.d, 1, d.norm_floor,
                                       h, st);
      if (rc) return rc;
    }
  } else if (d_encoder) {
    rc = launch_dict_rows<MODE_GRAD>(p, 0, p->b.encoder, p->dw_enc, nullptr, nullptr, d_encoder, rows, d.d, 1, d.norm_floor, h,
                                     st);
    if (rc) return rc;
  }
  if (p->b.encoder_bias && d_bias) {
    const long long tot = (long long)d.n_models * d.n;
    const int n_part = ((B + kBM - 1) / kBM) * 4;
    bias_kernel<MODE_GRAD><<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(
        p->b.encoder_bias, nullptr, nullptr, p->db_part, n_part, d.n, d.n_models, p->b.bias_decay, p->bnorm, d_bias, h,
        grad_out_scale(p, B), nullptr);
    CUDA_TRY(cudaGetLastError());
  }
  return SCE_OK;
}

int sce_step_host(sce_plan* p, const float* x_host, int B, float* out_losses_host, float* out_nnz_host,
                  void* stream) {
  if (!p) return fail(SCE_ERR_INVALID, "plan is NULL");
  if (!x_host) return fail(SCE_ERR_INVALID, "x_host is NULL");
  if (B < 1 || B > p->d.batch_max) return fail(SCE_ERR_INVALID, "B = %d outside [1, batch_max = %d]", B, p->d.batch_max);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t bytes = (size_t)input_models(p) * B * p->d.d * sizeof(float);
  CUDA_TRY(cudaMemcpyAsync(p->x_stage, x_host, bytes, cudaMemcpyHostToDevice, st));
  int rc = sce_step(p, p->x_stage, B, p->loss_stage, p->nnz_stage, st);
  if (rc) return rc;
  if (out_losses_host)
    CUDA_TRY(cudaMemcpyAsync(out_losses_host, p->loss_stage, (size_t)p->d.n_models * 4 * sizeof(float),
                             cudaMemcpyDeviceToHost, st));
  if (out_nnz_host)
    CUDA_TRY(cudaMemcpyAsync(out_nnz_host, p->nnz_stage, (size_t)p->d.n_models * sizeof(float), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  return SCE_OK;
}

int sce_read_code(sce_plan* p, int B, float* out_code, void* stream) {
  if (!p || !out_code) return fail(SCE_ERR_INVALID, "plan / out_code is NULL");
  if (B < 1 || B > p->d.batch_max) return fail(SCE_ERR_INVALID, "B = %d outside [1, batch_max = %d]", B, p->d.batch_max);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long per = (long long)B * p->d.n;
  for (int m = 0; m < p->d.n_models; ++m) {
    const long long src = (long long)m * p->d.batch_max * p->d.n;
    if (p->arith == kArithF16F8)
      join_code_kernel<kArithF16F8><<<1024, 256, 0, st>>>(p->c_hi + src, nullptr, p->c_x8 + src, out_code + (long long)m * per, per / 2);
    else
      join_code_kernel<kArithBf16x3><<<1024, 256, 0, st>>>(p->c_hi + src, p->c_lo + src, nullptr, out_code + (long long)m * per, per / 2);
  }
  CUDA_TRY(cudaGetLastError());
  return SCE_OK;
}

int sce_gather_rows(const void* chunk, int chunk_is_half, long long n_rows, int d, const long long* idx, int B,
                    const float* sub, float* out, void* stream) {
  if (!chunk || !out || B < 1 || d < 4 || d % 4) return fail(SCE_ERR_INVALID, "bad arguments to sce_gather_rows");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int blocks = (B + 7) / 8;
  if (chunk_is_half)
    gather_rows_kernel<__half><<<blocks, 256, 0, st>>>(static_cast<const __half*>(chunk), n_rows, d, idx, B, sub, out);
  else
    gather_rows_kernel<float><<<blocks, 256, 0, st>>>(static_cast<const float*>(chunk), n_rows, d, idx, B, sub, out);
  CUDA_TRY(cudaGetLastError());
  return SCE_OK;
}

int sce_last_launch_count(const sce_plan* plan) { return plan ? plan->last_launches : 0; }
int sce_input_absmax(sce_plan* plan, float* out_host, void* stream) {
  if (!plan || !out_host) return fail(SCE_ERR_INVALID, "plan / out_host is NULL");
  *out_host = 0.f;
  if (plan->arith != kArithF16F8) return SCE_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  uint32_t bits = 0;
  CUDA_TRY(cudaMemcpyAsync(&bits, plan->res_flags + kAbsmaxWord, sizeof(bits), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  memcpy(out_host, &bits, sizeof(bits));
  return SCE_OK;
}
int sce_health(sce_plan* plan, int* bad_out, float* absmax_out, void* stream) {
  if (!plan) return fail(SCE_ERR_INVALID, "plan is NULL");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  uint32_t words[kFlagWords];
  CUDA_TRY(cudaMemcpyAsync(words, plan->res_flags, sizeof(words), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  if (bad_out) *bad_out = words[kBadWord] != 0u;
  if (absmax_out) {
    *absmax_out = 0.f;
    if (plan->arith == kArithF16F8) memcpy(absmax_out, &words[kAbsmaxWord], sizeof(float));
  }
  return SCE_OK;
}
int sce_clear_health(sce_plan* plan, void* stream) {
  if (!plan) return fail(SCE_ERR_INVALID, "plan is NULL");
  CUDA_TRY(cudaMemsetAsync(plan->res_flags + kBadWord, 0, sizeof(uint32_t), static_cast<cudaStream_t>(stream)));
  return SCE_OK;
}

int sce_active_counts(sce_plan* plan, int B, int* counts, void* stream) {
  if (!plan || !counts) return fail(SCE_ERR_INVALID, "plan / counts is NULL");
  if (B < 1 || B > plan->d.batch_max) return fail(SCE_ERR_INVALID, "B = %d outside [1, batch_max = %d]", B, plan->d.batch_max);
  const int n_chunks = (plan->d.n + 31) / 32;
  active_count_kernel<<<dim3(n_chunks, plan->d.n_models), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      plan->act_pos, n_chunks, plan->d.batch_max, B, plan->d.n, counts);
  CUDA_TRY(cudaGetLastError());
  return SCE_OK;
}

int sce_plan_arith(const sce_plan* plan) {
  return !plan ? 0 : plan->arith == kArithF16F8 ? SCE_ARITH_F16F8 : SCE_ARITH_BF16X3;
}

int sce_profile_begin(sce_plan* p) {
  if (!p) return fail(SCE_ERR_INVALID, "plan is NULL");
  if (!p->prof_ev) {
    const int n = kProfMaxSteps * (SCE_PHASE_COUNT + 1);
    p->prof_ev = static_cast<cudaEvent_t*>(calloc(n, sizeof(cudaEvent_t)));
    if (!p->prof_ev) return fail(SCE_ERR_INVALID, "out of host memory");
    for (int i = 0; i < n; ++i) CUDA_TRY(cudaEventCreate(&p->prof_ev[i]));
  }
  p->prof_steps = 0;
  p->prof_on = true;
  return SCE_OK;
}

int sce_profile_end(sce_plan* p, float* phase_ms, int* steps_recorded) {
  if (!p || !phase_ms) return fail(SCE_ERR_INVALID, "plan / phase_ms is NULL");
  p->prof_on = false;
  for (int k = 0; k < SCE_PHASE_COUNT; ++k) phase_ms[k] = 0.f;
  for (int s = 0; s < p->prof_steps; ++s) {
    cudaEvent_t* ev = p->prof_ev + s * (SCE_PHASE_COUNT + 1);
    CUDA_TRY(cudaEventSynchronize(ev[SCE_PHASE_COUNT]));
    for (int k = 0; k < SCE_PHASE_COUNT; ++k) {
      float ms = 0.f;
      CUDA_TRY(cudaEventElapsedTime(&ms, ev[k], ev[k + 1]));
      phase_ms[k] += ms;
    }
  }
  if (steps_recorded) *steps_recorded = p->prof_steps;
  return SCE_OK;
}

long long sce_get_step_count(const sce_plan* plan) { return plan ? plan->step : 0; }
int sce_set_step_count(sce_plan* plan, long long steps_taken) {
  if (!plan || steps_taken < 0) return fail(SCE_ERR_INVALID, "bad arguments to sce_set_step_count");
  plan->step = steps_taken;
  return SCE_OK;
}

}  // extern "C"
