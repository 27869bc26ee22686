/*
 * lanpaint_b200 -- C ABI of the B200-native LanPaint Langevin hot path.
 *
 * The reference (scraed/LanPaint) is pure Python/PyTorch and has no FFI; this
 * header is the boundary a maintainer would bind (ctypes stub in
 * INTEGRATION.md).  Each entry point names the reference code it replaces,
 * paths relative to the reference root.
 *
 * Conventions
 *   - all tensors are fp32, contiguous, NC(T)HW; "per_sample" = C*spatial
 *   - the mask is uint8, 1 = known / keep (the reference's latent_mask,
 *     src/LanPaint/nodes.py:281-283), either full shape or [B,1,spatial]
 *     broadcast over channels (mask_channel_stride = 0)
 *   - per-sample scalars live in a device "coefficient table" of
 *     LP_TABLE_STRIDE floats per row, built on the host by
 *     lp_build_coef_table() -- this removes every exp/expm1/sqrt/where and
 *     every host sync of src/LanPaint/lanpaint.py:205,232-254,295-328 from
 *     the per-element path
 *   - every device entry point is asynchronous on the caller's stream, does
 *     not allocate, does not synchronise, is CUDA-graph capturable and
 *     re-entrant; it returns an lp_status (never throws)
 */
#ifndef LANPAINT_B200_H_
#define LANPAINT_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LP_ABI_VERSION 6
#define LP_TABLE_STRIDE 32 /* floats per table row (one 128-byte line), layout below */

typedef void* lp_stream_t; /* a cudaStream_t / CUstream */

typedef enum lp_status {
  LP_OK = 0,
  LP_ERR_INVALID = 1,   /* null pointer / negative size / bad flag combination */
  LP_ERR_ALIGNMENT = 2, /* reserved: all paths fall back to scalar access instead */
  LP_ERR_CUDA = 3,      /* launch failed; see lp_last_cuda_error() */
  LP_ERR_UNSUPPORTED = 4
} lp_status;

/* Table row layout (floats).  Class 0 = free / regenerate region ("x branch",
 * mask 0), class 1 = known region ("y branch", mask 1).
 *   0 c_tgt      sqrt(abt)/(1-abt)          coefficient of the score target in C
 *   1 S          model-space x = x_t * S    (VE: sqrt(1+sigma^2); flow: 1/(sqrt(abt)+sqrt(1-abt)))
 *   2 inv_S
 *   3 lam        Lambda
 *   4 one_plus_lam
 *   5 rep_noise  replace step: known = rep_noise*noise + rep_y*y
 *   6 rep_y
 *   7 corr       audio target correction c (1 = none)         [lanpaint.py:173-180]
 *   8+8k .. 15+8k  class k: g (= A - 1/(1-abt)), dt, e_full, k_full, sd_full, e_half, k_half, sd_half
 *   24,25      sdm[k]   = sqrt((e_half sd_half)^2 + sd_half^2): std of the two half-advance kicks a steady
 *                         fused launch applies, merged into one Gaussian (LP_SUBSTEP_MERGE_NOISE)
 *   26,27      sdmf[k]  = sqrt((e_half sd_full)^2 + sd_half^2): same for the FIRST|FUSE_NEXT launch
 *   28..31     reserved (0)
 * where for an advance over h:  e = exp(-A h), k = (1-e)/A, sd = sqrt(D^2 (1-exp(-2 A h))/(2A)), D = sqrt(2)
 * (src/LanPaint/lanpaint.py:232-254), full = dt, half = dt/2.
 */
enum {
  LP_T_CTGT = 0, LP_T_S = 1, LP_T_INVS = 2, LP_T_LAM = 3, LP_T_ONEPLAM = 4,
  LP_T_REPN = 5, LP_T_REPY = 6, LP_T_CORR = 7, LP_T_CLS0 = 8, LP_T_CLS1 = 16, LP_T_SDM = 24, LP_T_SDMF = 26,
  LP_C_G = 0, LP_C_DT = 1, LP_C_EF = 2, LP_C_KF = 3, LP_C_SF = 4, LP_C_EH = 5, LP_C_KH = 6, LP_C_SH = 7
};

/* Engine hyper-parameters: constructor of the reference engine,
 * src/LanPaint/lanpaint.py:8-21. */
typedef struct lp_hyper {
  double step_size;     /* StepSize */
  double lam;           /* Lambda */
  double beta;          /* Beta */
  double min_step_frac; /* MinStepFrac */
  int32_t flow;         /* IS_FLUX or IS_FLOW */
  int32_t reserved;
} lp_hyper;

typedef struct lp_dims {
  int64_t n_rows;              /* table rows == samples B (or B*2 with the audio class split) */
  int64_t per_row;             /* elements per table row (C*spatial for one sample) */
  int64_t spatial;             /* elements per channel */
  int64_t mask_row_stride;     /* mask elements between consecutive rows */
  int64_t mask_channel_stride; /* 0 = mask broadcast over channels, spatial = full-shape mask */
  int64_t row_split;           /* 0 = off.  > 0: positions >= row_split inside every row use table row
                                  (n_rows + row) instead of (row): the MiniMax-H3 flat pack, whose trailing
                                  audio positions run on their own sigma schedule (lanpaint.py:60-74); the
                                  table then holds 2*n_rows rows */
} lp_dims;

/* How the Gaussian draws of src/LanPaint/lanpaint.py:252 (torch.randn_like on
 * the global generator) are supplied. */
typedef enum lp_rng_mode {
  LP_RNG_TAPE = 0,   /* caller passes the draws as tensors (exact CPU-oracle parity) */
  LP_RNG_PHILOX = 1, /* in-kernel Philox4x32-10, element i <- component i&3 of counter (i>>2, draw) */
  LP_RNG_TORCH = 2   /* in-kernel Philox reproducing torch.randn_like's CUDA stream bit for bit */
} lp_rng_mode;

typedef struct lp_rng {
  int32_t mode;          /* lp_rng_mode */
  int32_t reserved;
  const float* tape0;    /* TAPE: draw consumed first by the launch */
  const float* tape1;    /* TAPE: draw consumed second (may be NULL if unused) */
  uint64_t seed;         /* PHILOX/TORCH */
  uint64_t draw0;        /* PHILOX: draw index; TORCH: philox offset of the first draw */
  uint64_t draw1;        /* second draw index / offset */
  const uint64_t* state; /* optional device pointer {seed, base}: if non-NULL, seed is read from
                            it and base is added to draw0/draw1 (lets a captured CUDA graph be
                            replayed with a fresh stream position) */
} lp_rng;

/* Element type of the model's output tensors ("heads").  State, clean latent, noise and all arithmetic are
 * fp32 like the reference's (its autocast(float32) wrappers, lanpaint.py:201,239); a network that returns
 * bf16 / fp16 predictions is read as is and widened in registers -- the same values the reference gets from
 * type promotion when it subtracts an fp32 x_t from them (lanpaint.py:182-184) -- instead of paying a
 * separate .float() pass (6 B/element read + 8 B/element written per head pair). */
typedef enum lp_dtype { LP_DTYPE_F32 = 0, LP_DTYPE_BF16 = 1, LP_DTYPE_F16 = 2 } lp_dtype;

/* The model's prediction(s) for one call, as the kernels consume them (src/LanPaint/lanpaint.py:34-43,
 * 159-171; src/LanPaint/nodes.py:161-175):
 *   combine == 0   a = x0, b = x0_BIG (NULL or == a: the two heads alias)
 *   combine != 0   a = cond, b = uncond (raw network outputs); the kernel forms
 *                  x0 = b + (a - b)*cfg and x0_BIG = b + (a - b)*cfg_big in registers with the eager
 *                  sub/mul/add roundings (requires dtype == LP_DTYPE_F32 so that they ARE the eager roundings) */
typedef struct lp_heads {
  const void* a;
  const void* b;
  int32_t dtype;   /* lp_dtype of a and b */
  int32_t combine;
  float cfg, cfg_big;
} lp_heads;

/* ---- library ---------------------------------------------------------- */
int lp_abi_version(void);
const char* lp_status_string(int status);
int lp_last_cuda_error(void); /* cudaError_t of the last failed launch on this thread */
/* Process-wide switches (also read once from the environment: LANPAINT_B200_PDL, LANPAINT_B200_TMA):
 *   "pdl" 1|0      programmatic dependent launch on every kernel (default 1)
 *   "tma" 1|0      use the TMA-staged persistent variants (cp.async.bulk + mbarrier ring) of the fused sub-step
 *                  (philox and torch streams) when eligible: at least 2^18 elements, spatial a multiple of 16,
 *                  no side outputs, no row split (default 1) */
int lp_set_option(const char* name, int value);

/* Host-only self test of the index arithmetic the kernels rely on (the multiply-shift division that
 * replaces `/` and `%` by per_row and spatial): returns the number of (n, d) pairs, out of `samples`
 * pseudo-random ones plus every edge case, for which it disagrees with n / d.  0 = sound. */
int64_t lp_selftest_index_math(int64_t samples);

/* Device self test of the FP32x2 (FFMA2) Box-Muller the torch-stream kernels use: runs it next to the scalar cuRAND
 * form on `n` pseudo-random input quadruples (plus 4096 edge cases: extremes of u and v, u == 1) and counts bitwise
 * mismatches into *mismatches_dev (a device uint64, zeroed by the call).  0 = the two are interchangeable. */
int lp_selftest_box_muller(int64_t n, uint64_t seed, unsigned long long* mismatches_dev, lp_stream_t stream);

/* ---- host: coefficient table ------------------------------------------- */
/* Replaces LanPaint.prepare_step_size + the mask blend of A/D/dt + the
 * exp/expm1/where/sqrt of advance_time_overdamped (lanpaint.py:81,205-214,
 * 232-254,295-328).  Inputs are the reference's own per-sample fp32 values
 * (abt, VE sigma: nodes.py:242-252) widened to double; arithmetic is fp64,
 * results rounded once to fp32.  rep_noise/rep_y may be NULL (-> 0, 1);
 * corr may be NULL (-> 1).  table_out: n_rows*LP_TABLE_STRIDE floats (host). */
int lp_build_coef_table(const double* abt, const double* ve_sigma, const double* rep_noise,
                        const double* rep_y, const double* corr, int64_t n_rows,
                        const lp_hyper* hyper, float* table_out);

/* Same table from explicit per-row half time steps (the `dtx/2`, `dty/2` a caller of the reference's
 * `langevin_dynamics(x_t, score, mask, step_size, current_times, sigma_x, sigma_y)` controls directly,
 * lanpaint.py:192,301-302).  scale = S per row (NULL: 1, i.e. the state stays in VP space).
 * target_is_x0e != 0: the kernels' x0 and y inputs both carry x_t + score (an arbitrary score callback's
 * result), so the known-region target must pass through unchanged (lam = 0 inside the target only). */
int lp_build_coef_table_dt(const double* abt, const double* scale, const double* dt_free,
                           const double* dt_known, double lam, int32_t target_is_x0e, int64_t n_rows,
                           float* table_out);

/* Geometry of torch's CUDA randn kernel (ATen/native/cuda/DistributionTemplates.h:
 * calc_execution_policy) for `numel` elements on `device`: grid blocks of 256
 * threads and the philox offset increment one draw consumes. */
int lp_torch_randn_geometry(int64_t numel, int device, int64_t* grid_out, uint64_t* increment_out);

/* ---- device: hot path --------------------------------------------------- */
/* mask_f32 > 0.5 -> uint8 (the binarise of nodes.py:281-283, done once). */
int lp_pack_mask_f32(const float* mask_f32, uint8_t* mask_u8, int64_t n, int invert, lp_stream_t stream);

/* Replace step + change of variables, lanpaint.py:85-99:
 *   x_model = mask ? rep_noise*noise + rep_y*y : x
 * written to x_model (may alias x) and, if non-NULL, x_copy. */
int lp_prologue_f32(const float* x, const float* y, const float* noise, const uint8_t* mask,
                    float* x_model, float* x_copy, const float* table, const lp_dims* dims,
                    lp_stream_t stream);

/* Flags of lp_substep_f32. */
enum {
  LP_SUBSTEP_FIRST = 1,     /* sub-step 0: no previous C, one full-dt advance (run_overdamped, args is None) */
  LP_SUBSTEP_FUSE_NEXT = 2, /* also apply the first half-advance of the NEXT sub-step (uses the new C) */
  LP_SUBSTEP_STORE_C = 4,   /* write the new C even without FUSE_NEXT (un-fused / early-stop loops) */
  LP_SUBSTEP_MERGE_NOISE = 8 /* with FUSE_NEXT and LP_RNG_PHILOX only: the two Gaussian kicks of the launch are
                                independent and nothing observes the state between them, so draw ONE normal with
                                the summed variance (table sdm/sdmf).  Same Markov chain in distribution, half the
                                RNG work; not stream-compatible with the reference, hence never used by TAPE/TORCH */
};

/* One fused Langevin launch = everything between two model calls
 * (lanpaint.py:113-142 -> langevin_dynamics :192-293 -> score_model :159-184,
 * Coef_C :217-220, advance_time_overdamped :232-254, run_overdamped :274-286):
 *   post-model half of sub-step i  [FIRST: C=Coef_C(x); x=adv(x,dt,C)
 *                                   else : Cn=Coef_C(x); x+=(Cn-C)dt; x=adv(x,dt/2,C_old)]
 *   + pre-model half of sub-step i+1 [x=adv(x,dt/2,Cn)] when FUSE_NEXT.
 * x_model is read (the model's input) and overwritten with the next model
 * input; c_state is read (unless FIRST) and written (FUSE_NEXT or STORE_C);
 * x0/x0_big are the model's two heads (x0_big NULL or == x0: aliased);
 * x_copy (optional) also receives the new x (the reference's
 * input_x.copy_(x), lanpaint.py:156); x0e_out (optional) receives
 * x_t + score, the LangevinState.x0 the early stopper watches.
 * Consumes 2 draws with FUSE_NEXT (1 with MERGE_NOISE), else 1. */
int lp_substep_f32(float* x_model, const float* x0, const float* x0_big, const float* y,
                   const uint8_t* mask, float* c_state, float* x_copy, float* x0e_out,
                   const float* table, const lp_dims* dims, const lp_rng* rng, int flags,
                   lp_stream_t stream);

/* The general form of lp_substep_f32: heads of any lp_dtype, optionally the two classifier-free-guidance
 * combines folded in (lp_heads).  lp_substep_f32 / lp_substep_cfg_f32 are this call with fp32 heads. */
int lp_substep(float* x_model, const lp_heads* heads, const float* y, const uint8_t* mask, float* c_state,
               float* x_copy, float* x0e_out, const float* table, const lp_dims* dims, const lp_rng* rng,
               int flags, lp_stream_t stream);

/* lp_substep_f32 with the two classifier-free-guidance combines folded in (SURVEY 8f rank 1; replaces the
 * two cfg_function calls of sampling_function_LanPaint, src/LanPaint/nodes.py:175): the caller passes the
 * network's raw cond / uncond x0 predictions and the two scales,
 *   x0 = uncond + (cond - uncond) * cfg ;   x0_big = uncond + (cond - uncond) * cfg_big
 * evaluated with the same three roundings as the eager sub/mul/add, so results equal the unfused path bit
 * for bit.  Same bytes read as lp_substep_f32; saves the 2 x 3 element-wise kernels and 2 tensors of
 * traffic the combines cost per model call. */
int lp_substep_cfg_f32(float* x_model, const float* cond, const float* uncond, float cfg, float cfg_big,
                       const float* y, const uint8_t* mask, float* c_state, float* x_copy, float* x0e_out,
                       const float* table, const lp_dims* dims, const lp_rng* rng, int flags,
                       lp_stream_t stream);

/* The un-fused building block: one exact OU advance of the model-space state,
 *   x_t = x/S;  x_t = e x_t + k C + sd xi;  x = x_t S
 * over dt (half = 0) or dt/2 (half = 1) -- advance_time_overdamped,
 * lanpaint.py:232-254.  Consumes 1 draw (rng->draw0 / tape0). */
int lp_advance_f32(float* x_model, const float* c_state, const uint8_t* mask, const float* table,
                   const lp_dims* dims, const lp_rng* rng, int half, lp_stream_t stream);

/* out = mask ? y : model_out   (lanpaint.py:151-154). */
int lp_epilogue_f32(const float* model_out, const float* y, const uint8_t* mask, float* out,
                    const lp_dims* dims, lp_stream_t stream);

/* lp_epilogue_f32 fused with the update k-diffusion's Euler sampler applies right after it
 * (sample_euler: d = (x - denoised)/sigma; x = x + d*(sigma_next - sigma)), for hosts that own the
 * sampler loop (SURVEY 8f rank 3):
 *   out = mask ? y : model_out ;  x = x + (x - out) * euler_coef      euler_coef = (sigma_next - sigma)/sigma
 * x_inout is the model-space state lp_substep_f32 left behind (the rewritten sampler x).  out may be NULL when
 * nobody reads the denoised latent (no preview callback): the pass then writes only x. */
int lp_epilogue_euler_f32(const float* model_out, const float* y, const uint8_t* mask, float* x_inout,
                          float* out, float euler_coef, const lp_dims* dims, lp_stream_t stream);

/* The boundary between two outer steps of a host-owned Euler loop in ONE pass: epilogue of step s
 * (lanpaint.py:151-154), k-diffusion's Euler update, and the replace step of step s+1 (lanpaint.py:85-94,
 * coefficients rep_noise/rep_y of `next_table`):
 *   out = mask ? y : model_out ;  x = x + (x - out)*euler_coef ;  x = mask ? rep_n*noise + rep_y*y : x
 * Known positions never read x or model_out; free positions never read noise.  out may be NULL. */
int lp_step_boundary_f32(const float* model_out, const float* y, const float* noise, const uint8_t* mask,
                         float* x_inout, float* out, float euler_coef, const float* next_table,
                         const lp_dims* dims, lp_stream_t stream);

/* The general boundary of an outer step, everything after its last model call in ONE pass
 * (lanpaint.py:151-157, k-diffusion sample_euler, lanpaint.py:85-94 of the next step):
 *   d   = model_out->combine ? b + (a - b)*cfg : a                      (heads of any lp_dtype)
 *   out = mask ? y : d                                                  written when out != NULL
 *   x   = x + (x - out)*euler_coef                                      when x_inout != NULL
 *   x   = mask ? rep_noise*noise + rep_y*y : x  (row of next_table)     when next_table != NULL (needs noise, x_inout)
 * lp_epilogue_f32, lp_epilogue_euler_f32, lp_step_boundary_f32 and lp_epilogue_cfg_f32 are special cases. */
int lp_boundary(const lp_heads* model_out, const float* y, const float* noise, const uint8_t* mask, float* x_inout,
                float* out, float euler_coef, const float* next_table, const lp_dims* dims, lp_stream_t stream);

/* Final denoise of an outer step straight from raw cond / uncond predictions:
 *   out = mask ? y : uncond + (cond - uncond)*cfg ;  if x_inout != NULL: x = x + (x - out)*euler_coef. */
int lp_epilogue_cfg_f32(const float* cond, const float* uncond, float cfg, const float* y, const uint8_t* mask,
                        float* x_inout, float* out, float euler_coef, const lp_dims* dims, lp_stream_t stream);

/* Early-stop statistics (LanPaintEarlyStopper, src/LanPaint/earlystop.py:32-55,238-313):
 *   sums[0] = sum over elements with mask == 0 (the inpaint weight)  of (scale*(a-b))^2
 *   sums[1] = sum over elements with ring != 0 (4-neighbour boundary) of (scale*(a-b))^2
 * i.e. the numerators of _weighted_mse for the inpaint and boundary-ring weights; the denominators are
 * constants of the mask.  ring may be NULL (sums[1] = 0); table may be NULL (scale = 1), otherwise
 * scale = inv_S of the row, which turns a model-space difference into the VP-space one the reference
 * measures on x_t.  ring uses the mask's layout/strides.  sums: 2 doubles on the device, zeroed by the call.
 * Warp-shuffle + one atomicAdd(double) per block per sum. */
int lp_stop_stats_f32(const float* a, const float* b, const uint8_t* mask, const uint8_t* ring,
                      const float* table, const lp_dims* dims, double* sums, lp_stream_t stream);

/* ---- device: utilities (tests, bench) ---------------------------------- */
/* out[i] ~ N(0,1) with the given rng (PHILOX or TORCH; draw0 only). */
int lp_fill_normal_f32(float* out, int64_t n, const lp_rng* rng, lp_stream_t stream);

/* The noise image of a sample call with the bits of ComfyUI's CPU draw.  `comfy.sample.prepare_noise`, which
 * nodes.common_ksampler calls for every LanPaint KSampler node (src/LanPaint/nodes.py:513,589), is
 * `torch.manual_seed(seed); torch.randn(size, generator=..., device="cpu")`: at::mt19937 (one 32-bit output per
 * float, 24 bits kept), torch's normal_fill (Box-Muller over the pairs (j, j+8) of every 16 values; a size that is
 * not a multiple of 16 redraws its last 16) with avx_mathfun.h's cephes log / sincos as the AVX2 build executes them.
 * Writes out[0..n) ~ N(0,1) with exactly those bits (fp32, n >= 16; `out` must have room for n + 16 floats).
 * state_out (optional, 624 words on the device) receives the generator's state array after its last twist and
 * *consumed_out (optional, host) the number of 32-bit outputs drawn, so that the caller can leave the host's CPU
 * generator where ComfyUI's own call would have left it.  One CTA walks the (sequential) generator; the transform
 * is a second, parallel launch. */
int lp_torch_cpu_randn_f32(float* out, int64_t n, uint64_t seed, uint32_t* state_out, int64_t* consumed_out,
                           lp_stream_t stream);

/* Synthetic pointwise two-head denoiser used by bench.py (SURVEY 8d):
 *   h0 = a0*x + b0*tanh(x) + c0 ;  h1 = a1*x + c1     coef = {a0,b0,c0,a1,c1} */
int lp_synth_denoiser_f32(const float* x, float* h0, float* h1, int64_t n, const float* coef5_host,
                          lp_stream_t stream);
/* Same, heads written in `dtype` (a network that computes in bf16 returns bf16 predictions). */
int lp_synth_denoiser(const float* x, void* h0, void* h1, int dtype, int64_t n, const float* coef5_host,
                      lp_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* LANPAINT_B200_H_ */
