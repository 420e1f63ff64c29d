// kernels.cuh — host launchers of the CUDA-core kernels (kernels_simt.cu, kernels_embed.cu,
// kernels_step.cu).  T is the activation storage type: float (fp32 mode) or __nv_bfloat16.
#pragma once
#include "common.cuh"

namespace tcs {

// ---- embeddings (kernels_embed.cu) -----------------------------------------------------
struct EmbedWeights {           // device pointers into the fp32 weight arena (PyTorch layouts)
  const float *cat_emb;         // [n_types+1,128]
  const float *cm0_w, *cm0_b;   // cond_emb.cont_mlp.0  [128,ycd],[128]
  const float *cm2_w, *cm2_b;   // cond_emb.cont_mlp.2  [128,128]
  const float *co_w, *co_b;     // cond_emb.out.1       [128,256]
  const float *tm0_w, *tm0_b;   // time_mlp.0           [128,128]
  const float *tm2_w, *tm2_b;   // time_mlp.2
  const float *tc_w, *tc_b;     // to_cond_map          [8,128]
  const float *tt_w, *tt_b;     // to_time_map          [8,128]
  const float *wsum;            // [96][16]  sum over the 9 taps of down1.net.0.weight[:,1+c]
  const float *b0;              // down1.net.0.bias [96]
  int n_types, y_cont_dim;
};
// cvec[b][96]: condition part of the folded first-conv bias.  nb rows; row r uses sample
// r/dup of (y_cat,y_cont) and is the unconditional (null token, zeros) row when dup==2 && r odd.
int launch_cond_embed(const EmbedWeights& w, const int64_t* y_cat, const float* y_cont, int n, int dup, float* cvec,
                      cudaStream_t st);
// tvec[r][96] = down1.net.0.bias + time part, for nt time values
int launch_time_embed(const EmbedWeights& w, const float* t, int nt, float* tvec, cudaStream_t st);

// ---- first conv: 1 -> 96, 3x3 circular, bias = tvec[trow] + cvec[b] -------------------------
// x [n,64,64]; raw [n*dup,64,64,96]; partials [n*dup][32][8][2] (32 slots per image)
int launch_first_conv(const float* x, const float* w9 /*[96][9]*/, const float* tvec, int tvec_stride,
                      const int* step_ptr, int trow_off, const float* cvec, int n, int dup, float* raw,
                      float* partials, cudaStream_t st);
constexpr int FIRST_CONV_SLOTS = 32;
// the same conv with GroupNorm(down1.net.1)+SiLU fused: x -> padded T [n*dup,66,66,96] (no fp32 round trip)
template <typename T>
int launch_first_conv_gn(const float* x, const float* w9, const float* tvec, int tvec_stride, const int* step_ptr,
                         int trow_off, const float* cvec, int n, int dup, const float* gamma, const float* beta, T* out,
                         cudaStream_t st);

// ---- GroupNorm apply (+SiLU) -> padded T with halo -----------------------------------------
// in: fp32 raw plain [B,H,W,C] (in_padded=0) or padded T (in_padded=1); partials [B][slots][8][2]
template <typename T>
int launch_gn_apply(const void* in, int in_padded, const float* partials, int slots, const float* gamma,
                    const float* beta, int B, int H, int W, int C, int silu, T* out_padded, float2* stats_scratch /*[B][8]*/,
                    cudaStream_t st);
// GroupNorm (no activation) of padded 16x16x192 images in one kernel: padded T -> padded T (attn.norm)
template <typename T>
int launch_gn_image16(const T* in_padded, int B, const float* gamma, const float* beta, T* out_padded, cudaStream_t st);
// statistics of a padded T tensor -> partials [B][1][8][2]
template <typename T>
int launch_gn_stats(const T* in_padded, int B, int H, int W, int C, float* partials, cudaStream_t st);

// ---- bilinear x2 (align_corners=False, edge clamp): padded T [B,h+2,w+2,C] -> padded [B,2h+2,2w+2,C]
template <typename T>
int launch_upsample2x(const T* in, int B, int h, int w, int C, T* out, cudaStream_t st);

// ---- attention: qkv plain T [B,256,576] -> y plain T [B,256,192] ----------------------------
template <typename T>
int launch_attention(const T* qkv, int B, T* y, cudaStream_t st);

// ---- generic SIMT conv (fp32 accumulate), same epilogues as the tensor-core engine ------------
// weights packed fp32 [k*k][cin_total][ntot]
template <typename T>
int launch_conv_simt(const ConvGeom& g, const T* src0, const T* src1, const float* wpacked, int epi,
                     const EpiArgs& ea, cudaStream_t st);
void conv_simt_pack_weights(const ConvGeom& g, const float* w, float* out_host, bool round_bf16);

// ---- out conv 96 -> 1 with the CFG combine in its epilogue -----------------------------------
// act padded T [n*dup,66,66,96]; eps [n,64,64] = dup==2 ? e_u + s(e_c - e_u) : e
template <typename T>
int launch_out_conv(const T* act, const float* w /*[9][96]*/, float bias, int n, int dup, float guidance,
                    float* eps, cudaStream_t st);

// ---- layout helpers (debug hooks / tests) ------------------------------------------------------
template <typename T>
int launch_pad_from_plain(const float* in, int B, int H, int W, int C, int pad, T* out, cudaStream_t st);
template <typename T>
int launch_unpad_to_f32(const T* in, int B, int H, int W, int C, int pad, float* out, cudaStream_t st);

// ---- fp32 mode on the tensor pipe: bf16 (hi, lo) split tensors (kernels_split.cu) ------------------------------------
// split tensor = hi plane, then the lo plane lo_off elements later; a ~= hi + lo to ~2^-17 relative
int launch_split(const float* in, size_t elems, __nv_bfloat16* out, size_t lo_off, cudaStream_t st);
// raw fp32 conv output [B,H,W,C] -> padded tensor with halo.  mode 0: GroupNorm(stats) + SiLU -> split tensor;
// mode 1: copy -> split tensor; mode 2: + residual (padded fp32) -> padded fp32
int launch_raw_to_padded(int mode, const float* raw, const float2* stats, const float* gamma, const float* beta,
                         const float* residual, int B, int H, int W, int C, void* out, size_t lo_off, cudaStream_t st);
int launch_unsplit_to_f32(const __nv_bfloat16* in, size_t lo_off, int B, int H, int W, int C, int pad, float* out,
                          cudaStream_t st);
// stats[b][g] = (mean, rstd) from the convs' partial sums (fp64 combine, fixed order)
int launch_gn_finalize(const float* partials, int slots, int B, int H, int W, int C, float2* stats, cudaStream_t st);

// ---- sampler update (kernels_step.cu) ------------------------------------------------------------
struct StepCoef {   // one row per time-grid index i (host-computed in fp32, see tcs_api.cu)
  float t, beta, sigma, alpha, dt, g_sqrt_dt, pad0, pad1;   // dt = ts[i+1]-ts[i]; g_sqrt_dt = sqrt(beta)*sqrt(|dt|)
};
// DPM-Solver++(2M) row i (host-computed in double from the fp32 log-SNR grid, each rounded to fp32 once):
// a = sigma_{i+1}/sigma_i, m = alpha_{i+1}*(-expm1(-h_i)), D = c0*x0 + c1*x0_prev; c1 == 0 marks a first-order row
struct DpmCoef {
  float a, m, c0, c1;
};
enum StepMode : int { STEP_SDE = 0, STEP_ODE_PREDICT = 1, STEP_ODE_CORRECT = 2, STEP_FINAL = 3, STEP_DPM2M = 4 };
struct StepArgs {
  const StepCoef* coef;     // device table
  const DpmCoef* dpm;       // DPM2M: device table beside `coef`, same row index
  const int* step_ptr;      // device step counter (row = *step_ptr + row_off)
  int row_off;
  int mode;
  float* x;                 // [n,4096] state (read; written for SDE / ODE_CORRECT / DPM2M)
  float* x_pred;            // ODE: Euler predictor state
  float* d0;                // ODE: first drift; DPM2M: x0_prev (the data prediction of the previous step)
  const float* eps;         // [n,4096]
  const float* noise;       // injected z for all steps [steps,n_total,4096] or null -> Philox
  long long noise_step_stride;  // elements between consecutive steps in `noise`
  float* out_img;           // FINAL: [n,4096] in [0,1]
  float* out_x0;            // FINAL: optional pre-clamp x0_hat
  unsigned long long seed, gidx0;  // Philox key / global index of sample 0 of this launch
  int n;
};
int launch_step(const StepArgs& a, cudaStream_t st);
// x[i] ~ N(0,1) keyed (seed, gidx0+i, counter word 0)
int launch_philox_normal(float* x, int n, unsigned long long seed, unsigned long long gidx0, cudaStream_t st);
int launch_advance(int* step_ptr, int delta, cudaStream_t st);
int launch_copy_f32(float* dst, const float* src, size_t n, cudaStream_t st);

}  // namespace tcs
