// linear_tc.cuh — host interface of the tcgen05 GEMM used by the latent diffusion prior (linear_tc.cu):
//   out[M,N] = act(A[M,K] · W[N,K]^T + bias)     A, W bf16 K-major (W is the nn.Linear weight layout), fp32 accumulate.
#pragma once
#include "common.cuh"

namespace tcs {

enum LinFlags : int {
  LIN_SILU = 1,        // SiLU on (acc + bias)
  LIN_OUT_F32 = 2,     // fp32 output (default bf16)
  LIN_ACCUM = 4,       // fp32 output only: out += acc + bias (the residual stream h of the FiLM blocks)
  LIN_RELU_TC = 8      // ReLU on (acc + bias) (decoder)
};

struct LinearTcParams {
  int M, N, K;
  int n_mtiles, n_ntiles, kblocks;   // 128-row M tiles (padded to an even count for CTA pairs), 256-col N tiles, K/64
  int nstage;
  uint32_t a_bytes, stage_bytes;
  const float* bias;                 // [N] or null
  void* out;
  int ldo;                           // elements between output rows
  int flags;
  // transposed-convolution mode (linear_tc_make_convt_plan): M tiles are windows of the NHWC input
  int Hi, n_img, cblocks;            // input size, images, 64-channel blocks per tap (kblocks = 4 * cblocks)
  int tiles_per_img, rows_y, imgs;   // M tile = `imgs` whole images (Hi*Hi < 128) or `rows_y` rows of one image
};

struct LinearTcPlan {
  CUtensorMap mapA, mapW, mapO;
  LinearTcParams p;
  int bn;        // N tile: 256 (Linear) or C_out (transposed conv: 128 / 64 / 32)
  bool conv = false;
  int grid;
  size_t smem;
  bool valid = false;
};

// A: bf16 [M, K] with row pitch lda elements; W: bf16 [N, K] with row pitch ldw elements (both 16-byte aligned pitches).
// Needs N % 256 == 0 and K % 64 == 0; M is arbitrary (TMA zero-fills, the epilogue masks).
int linear_tc_make_plan(LinearTcPlan* plan, const __nv_bfloat16* A, int lda, const __nv_bfloat16* W, int ldw, int M, int N,
                        int K, const float* bias, void* out, int ldo, int flags, int sm_count);
// ConvTranspose2d(C_in -> C_out, k 4, s 2, p 1) + ReLU: in bf16 NHWC [n, Hi, Hi, C_in] -> out bf16 NHWC [n, 2Hi, 2Hi, C_out].
// wpacked bf16 [4 parity][C_out][4 taps * C_in] (vae_convt_pack_weights order), bias fp32 [C_out].
// Needs Hi in {4, 8, 16}, C_in % 64 == 0, C_out in {32, 64, 128}.
int linear_tc_make_convt_plan(LinearTcPlan* plan, const __nv_bfloat16* in, const __nv_bfloat16* wpacked, const float* bias,
                              int n, int Hi, int Ci, int Co, __nv_bfloat16* out, int sm_count);
int linear_tc_launch(const LinearTcPlan& plan, cudaStream_t st);

}  // namespace tcs
