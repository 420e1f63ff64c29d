/*
 * tcs.h — C ABI of libtcs.so, the B200 (sm_100a) ToyCrystals score-sampler library.
 *
 * The reference (sahhermans/vae-diffusion-toy-crystals) is pure Python and has no FFI; the
 * boundary a maintainer would bind is therefore the set of Python callables on the sampling
 * path.  Each entry point below names the reference interface it replaces
 * (paths relative to the reference root):
 *
 *   tcs_create / tcs_set_weight / tcs_finalize_weights / tcs_destroy
 *        <- CondUNetTiny.__init__ + load_state_dict     src/toycrystals/models/sde_score_model.py:180-225
 *           checkpoint reader                            scripts/sample_sde_score_model.py:67-105
 *   tcs_score
 *        <- CondUNetTiny.forward  (:243-266)  and  predict_eps_cfg (:402-423)
 *   tcs_sample
 *        <- sample_probability_flow_ode (:452-504), sample_reverse_sde_euler_maruyama (:507-569),
 *           VPSDE (:273-298); also DPM-Solver++(2M) and SDE-DPM-Solver++(2M), which the reference does not have
 *   tcs_condition_grid
 *        <- save_sde_samples condition synthesis (:317-321)
 *
 * Conventions: plain C types only.  All tensor pointers are DEVICE pointers unless the name
 * ends in _host.  Images are [n,1,64,64] fp32 contiguous (C==1 so NCHW == NHWC).  The caller
 * owns every buffer it passes and must keep it alive until the work enqueued on `stream`
 * has completed.  Work is asynchronous on `stream` (a cudaStream_t cast to void*; NULL =
 * legacy default stream).  A handle is bound to one device and is not re-entrant.
 * Every function returns 0 on success or a negative tcs_status; the message is available
 * from tcs_last_error() (thread local).  There is no CPU fallback anywhere in this library.
 */
#ifndef TCS_H_
#define TCS_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct tcs_handle tcs_handle;

enum tcs_status {
  TCS_OK = 0,
  TCS_ERR_BAD_ARGUMENT = -1,   /* maps to ValueError in the Python shim            */
  TCS_ERR_UNSUPPORTED = -2,    /* legal reference config this build does not cover */
  TCS_ERR_CUDA = -3,           /* CUDA runtime / driver failure                    */
  TCS_ERR_STATE = -4           /* e.g. sampling before tcs_finalize_weights        */
};

enum tcs_precision { TCS_FP32 = 0, TCS_BF16 = 1 };
enum tcs_engine { TCS_ENGINE_AUTO = 0, TCS_ENGINE_SIMT = 1, TCS_ENGINE_TCGEN05 = 2 };
/* ODE: probability-flow ODE, Heun, quadratic time grid.  SDE: reverse VP-SDE, Euler-Maruyama.
 * DPMPP_2M: DPM-Solver++(2M) (Lu et al. 2022, Algorithm 2) on the probability-flow ODE, times uniform in
 *           log-SNR, one evaluation per step, deterministic (noise must be NULL).  Not in the reference.
 * DPMPP_2M_SDE: SDE-DPM-Solver++(2M) (Lu et al. 2022, the SDE variant of Algorithm 2, eta = 1) on the reverse VP-SDE: the
 *           same grid and (c0, c1) as DPMPP_2M, one evaluation per step, stochastic: z per step from `noise` or from
 *           Philox keyed (seed, global sample index, 1 + step), as for SDE.  Not in the reference. */
enum tcs_sampler { TCS_SAMPLER_ODE = 0, TCS_SAMPLER_SDE = 1, TCS_SAMPLER_DPMPP_2M = 2, TCS_SAMPLER_DPMPP_2M_SDE = 3 };

typedef struct tcs_config {
  int32_t n_types;     /* CondUNetTiny(n_types, ...)                                  */
  int32_t y_cont_dim;
  int32_t base_ch;     /* only 96 is supported (reference CLI default / README model) */
  int32_t emb_dim;     /* only 128 */
  int32_t cond_ch;     /* only 8   */
  int32_t time_ch;     /* only 8   */
  double beta_min;     /* VPSDE(beta_min, beta_max); doubles, as the Python floats are */
  double beta_max;
  int32_t precision;   /* tcs_precision: activation/weight storage of the conv operands */
  int32_t engine;      /* tcs_engine: AUTO = tcgen05 for bf16, SIMT (FFMA) for fp32     */
  int32_t device;      /* CUDA ordinal */
  int32_t chunk;       /* images per network pass (0 = library default); sizing knob only */
  int32_t use_graph;   /* 1 = replay the per-step launch sequence from a CUDA graph      */
  int32_t fuse_gn;     /* 1 (default) = GroupNorm+SiLU fused into the tcgen05 conv epilogue (pre-norm values are staged as
                          fp16: |v| <= 65504); 0 = conv -> fp32 -> GroupNorm kernel, any magnitude */
} tcs_config;

/* Fill *cfg with the reference defaults (n_types 4, y_cont_dim 4, 96/128/8/8, beta 0.1..30). */
void tcs_default_config(tcs_config* cfg);

int tcs_create(tcs_handle** out, const tcs_config* cfg);
void tcs_destroy(tcs_handle* h);

/* One call per state-dict entry, key spelled as in CondUNetTiny.state_dict().  `data` is fp32,
 * contiguous, host or device memory (copied before the call returns). */
int tcs_set_weight(tcs_handle* h, const char* key, const float* data, const int64_t* shape, int32_t ndim);

/* Validates that all 71 tensors arrived with the right shapes, packs them for the kernels. */
int tcs_finalize_weights(tcs_handle* h);

/* eps_hat for one network evaluation.
 *   x       [n,1,64,64]        t [n] (per-sample times, as CondUNetTiny.forward allows)
 *   y_cat   [n] int64          y_cont [n,y_cont_dim]
 *   guidance <= 0 : eps = net(x,t,y_cat,y_cont)
 *   guidance  > 0 : eps = eps_u + guidance*(eps_c - eps_u), both branches in one doubled batch
 *   eps_out [n,1,64,64] */
int tcs_score(tcs_handle* h, const float* x, const float* t, const int64_t* y_cat, const float* y_cont,
              int32_t n, float guidance, float* eps_out, void* stream);

typedef struct tcs_sample_args {
  int32_t sampler;              /* tcs_sampler */
  int32_t n;                    /* samples produced by this call */
  int32_t steps;
  float guidance;
  double t_end;                 /* must lie in (0,1) */
  const int64_t* y_cat;         /* [n] */
  const float* y_cont;          /* [n,y_cont_dim] */
  const float* x_init;          /* [n,1,64,64] or NULL -> Philox N(0,1) */
  const float* noise;           /* [steps,n,1,64,64] or NULL -> Philox N(0,1) (SDE, DPMPP_2M_SDE; NULL for DPMPP_2M) */
  uint64_t seed;                /* Philox key */
  uint64_t global_index_offset; /* index of sample 0 of this call in the whole job (sharding) */
  float* x_out;                 /* [n,1,64,64] images in [0,1] */
  float* trace_eps;             /* NULL or [nfe,n,1,64,64]: CFG-combined eps of every evaluation */
  float* trace_x;               /* NULL or [nfe,n,1,64,64]: the x_t every evaluation saw */
  float* x0_hat;                /* NULL or [n,1,64,64]: projection before the [0,1] map/clamp */
  double beta_min;              /* VPSDE(beta_min, beta_max) of THIS call; beta_max <= 0 -> the tcs_config values. */
  double beta_max;              /* (The schedule is per call, as in the reference where `sde` is a sampler argument.) */
} tcs_sample_args;

int tcs_sample(tcs_handle* h, const tcs_sample_args* args, void* stream);

/* Number of network evaluations tcs_sample performs: ode (Heun) 2*steps+1, sde, dpm++2m and dpm++2m-sde steps+1. */
int32_t tcs_nfe(int32_t sampler, int32_t steps);

/* y_cat[i] = (offset+i) % n_types ; y_cont[i] = [0, theta_max*(offset+i)/(n_total-1), 0, ...]. */
int tcs_condition_grid(tcs_handle* h, int32_t n, int64_t offset, int64_t n_total, float theta_max,
                       int64_t* y_cat, float* y_cont, void* stream);

/* The fused VP-SDE update on its own (the kernel the HBM roofline is quoted for):
 *   x <- x + (-0.5 b x + b eps / sigma) dt + sqrt(b) sqrt(|dt|) z    (sampler = SDE)
 * z from `noise` (may be NULL -> Philox keyed (seed, global index, step)). */
int tcs_sde_update(tcs_handle* h, float* x, const float* eps, const float* noise, int32_t n, float t, float t_next,
                   uint64_t seed, uint64_t global_index_offset, int32_t step, void* stream);

/* The probability-flow (Heun) update kernels on their own (sde_score_model.py:426-449, :490-493, :496-504), for the
 * bit-exactness tests.  mode 1 = predictor: d0 <- drift(x, eps, t), x_pred <- x + d0 * (t_next - t);
 * mode 2 = corrector: x <- x + 0.5 * (d0 + drift(x_pred, eps, t_next)) * (t_next - t);
 * mode 3 = final projection at t: x0_hat <- (x - sigma eps) / max(alpha, 1e-6) into d0, image into x_pred. */
int tcs_ode_update(tcs_handle* h, int32_t mode, float* x, float* x_pred, float* d0, const float* eps, int32_t n,
                   float t, float t_next, void* stream);

/* The DPM-Solver++(2M) update kernel on its own (bit-exactness tests), in fp32 and in this order:
 *   x0 = (x - sigma*eps)/alpha;  D = c1 == 0 ? x0 : c0*x0 + c1*x0_prev;  x <- a*x + m*D;  x0_prev <- x0
 * (c1 == 0 is a first-order row: x0_prev is not read). */
int tcs_dpm_update(tcs_handle* h, float* x, float* x0_prev, const float* eps, int32_t n, float alpha, float sigma, float a,
                   float m, float c0, float c1, void* stream);

/* The SDE-DPM-Solver++(2M) update kernel on its own (bit-exactness tests), in fp32 and in this order:
 *   x0 = (x - sigma*eps)/alpha;  D = c1 == 0 ? x0 : c0*x0 + c1*x0_prev;  x <- (a*x + m*D) + g*z;  x0_prev <- x0
 * z from `noise` [n,1,64,64] (this step only), or NULL -> Philox keyed (seed, global_index_offset + i, 1 + step). */
int tcs_dpm_sde_update(tcs_handle* h, float* x, float* x0_prev, const float* eps, const float* noise, int32_t n,
                       float alpha, float sigma, float a, float m, float c0, float c1, float g, uint64_t seed,
                       uint64_t global_index_offset, int32_t step, void* stream);

/* Host-side schedule, exactly as the kernels use it (for tests): ts has steps+1 entries. */
int tcs_time_grid_host(int32_t steps, double t_end, float* ts_host);
int tcs_schedule_host(double beta_min, double beta_max, float t, float* beta, float* alpha, float* sigma);
/* The DPM-Solver++(2M) schedule tcs_sample uses (steps >= 1): ts_host [steps+1] = times uniform in
 * log-SNR lambda = log alpha - log sigma from t = 1 to t_end (endpoints exact), fp32; coef_host [steps][4] =
 * (a, m, c0, c1) of every step, computed in double from the fp32 times and rounded once:
 *   h = lambda(t_{i+1}) - lambda(t_i), a = sigma(t_{i+1})/sigma(t_i), m = alpha(t_{i+1})*(-expm1(-h)),
 *   (c0, c1) = (1, 0) on step 0 and, when steps < 15, on the last step; else r = h_{i-1}/h_i, (1 + 1/(2r), -1/(2r)). */
int tcs_dpm_schedule_host(int32_t steps, double t_end, double beta_min, double beta_max, float* ts_host,
                          float* coef_host);
/* The SDE-DPM-Solver++(2M) schedule: the same ts_host and (c0, c1) as tcs_dpm_schedule_host; coef_host [steps][5] =
 * (a, m, c0, c1, g), in double from the fp32 times and rounded once:
 *   a = sigma(t_{i+1})/sigma(t_i) * exp(-h), m = alpha(t_{i+1})*(-expm1(-2h)), g = sigma(t_{i+1})*sqrt(-expm1(-2h)). */
int tcs_dpm_sde_schedule_host(int32_t steps, double t_end, double beta_min, double beta_max, float* ts_host,
                              float* coef_host);

/* Waits for the handle's enqueued work and returns its sticky status bits (then clears them):
 *   bit 0: a fused GroupNorm layer saw a pre-norm activation that may exceed the fp16 staging range; the eps / images of
 *          the calls since the last check are INVALID - re-run with tcs_config.fuse_gn = 0 (the Python shim does).
 * Negative = tcs_status (e.g. a kernel fault). */
int32_t tcs_check(tcs_handle* h);
/* bit 0: GroupNorm fused into the conv epilogue; bit 1: fused layers launch as CTA pairs with the cooperative attribute;
 * bits 8..: CTAs of the fused kernel the device holds at once (cudaOccupancyMaxActiveClusters * 2). */
int32_t tcs_launch_mode(const tcs_handle* h);

/* Counters: kernels launched by this handle since creation / library build info. */
int64_t tcs_launch_count(const tcs_handle* h);
const char* tcs_build_info(void);
const char* tcs_last_error(void);

/* ---- test hooks (used by tests/ only; stable enough to bind, not part of the drop-in) ---- */
/* Run one network pass and copy the named internal activation (NHWC fp32, unpadded) to `out`.
 * names: "down1.net.0.raw", "down1.net.3.raw", "ds1", ... as in oracle taps.  Returns the
 * number of floats written (or a negative status). */
int64_t tcs_debug_layer(tcs_handle* h, const char* name, const float* x, const float* t, const int64_t* y_cat,
                        const float* y_cont, int32_t n, int32_t uncond, float* out, int64_t out_capacity,
                        void* stream);

/* tcs_score for one network pass (n * (guidance > 0 ? 2 : 1) <= chunk images) with CUDA events recorded, on the
 * library's own stream, around every tensor-core conv launch.  conv_ms[15] is in execution order: down1.net.3,
 * ds1, down2.net.0, down2.net.3, ds2, mid.net.0, mid.net.3, attn.qkv, attn.proj, us2_conv, up2.net.0, up2.net.3,
 * us1_conv, up1.net.0, up1.net.3 (GroupNorm+SiLU included where fused); *total_ms = the whole pass.  Synchronous. */
int tcs_score_profiled(tcs_handle* h, const float* x, const float* t, const int64_t* y_cat, const float* y_cont,
                       int32_t n, float guidance, float* eps_out, float* conv_ms_host, float* total_ms_host,
                       void* stream);

/* Run ONE convolution layer in isolation (synchronous; allocates its own scratch).
 *   in0/in1 : fp32 NHWC [B, H_out*stride, W_out*stride, cin] (in1 may be NULL when cin1 == 0)
 *   weight  : [cout, cin0+cin1, k, k] (PyTorch layout), bias [cout]
 *   epi     : 0 raw fp32 + GroupNorm partial sums, 1 padded (halo) output, 2 plain output
 *   out     : fp32 NHWC [B,H_out,W_out,cout];  stats: NULL or [B,8,2] = per-group (sum, sum of squares)
 * engine/precision as in tcs_config (tcgen05 needs bf16). */
int tcs_debug_conv(int32_t engine, int32_t precision, int32_t B, int32_t H_out, int32_t W_out, int32_t cin0,
                   int32_t cin1, int32_t cout, int32_t ksize, int32_t stride, const float* in0, const float* in1,
                   const float* weight, const float* bias, float* out, float* stats, int32_t epi, void* stream);

/* us1_conv / us2_conv with the bilinear x2 upsample fused into the conv (tcgen05 engine, bf16): in_lowres is fp32 NHWC
 * [B, H_out/2, W_out/2, cin]; out = conv3x3_circular(upsample_bilinear_x2(in_lowres)) + bias, fp32 NHWC [B,H_out,W_out,cout]
 * (nn.Upsample + nn.Conv2d(padding_mode="circular"), sde_score_model.py:217-222,256-262).  Synchronous. */
int tcs_debug_conv_ups(int32_t B, int32_t H_out, int32_t W_out, int32_t cin, int32_t cout, const float* in_lowres,
                       const float* weight, const float* bias, float* out, void* stream);

/* Host-only helper of the tests: the byte image of the attention block's weights as attn_block_tc_kernel copies it into
 * shared memory (host pointers: qkv_w [576,192], proj_w [192,192]): per head [3 blocks of 64 input channels][144 rows =
 * q | k | v rows of the head][128 B], then the projection [3][192 rows][128 B]; bf16, every 128-byte row with its 16-byte
 * chunks at (chunk ^ (row & 7)) = SWIZZLE_128B.  out == NULL returns the size in bytes. */
int64_t tcs_debug_attn_pack(const float* qkv_w, const float* proj_w, uint8_t* out, int64_t capacity);

/* Run the fused attention block (csrc/attn_tc.cu: GroupNorm -> qkv -> softmax(q k^T / sqrt(48)) v -> proj -> + x,
 * SelfAttention2d.forward, sde_score_model.py:136-167) in isolation, bf16 / tcgen05.  Device fp32 pointers:
 *   x, out  : NHWC [B,16,16,192];  gn_w, gn_b [192];  qkv_w [576,192], qkv_b [576];  proj_w [192,192], proj_b [192]
 *   dbg     : NULL, or 246784 floats receiving intermediates of image 0: normalised input [256][192], q|k|v + bias
 *             [256][576], attention output [256][192], softmax denominators (base-2 scaled) [256][4].  Synchronous. */
int tcs_debug_attn_block(int32_t B, const float* x, const float* gn_w, const float* gn_b, const float* qkv_w,
                         const float* qkv_b, const float* proj_w, const float* proj_b, float* out, float* dbg,
                         void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TCS_H_ */