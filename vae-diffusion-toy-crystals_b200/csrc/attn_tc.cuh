// attn_tc.cuh — host interface of the fused SelfAttention2d block on tcgen05 (attn_tc.cu).
#pragma once
#include "common.cuh"

namespace tcs {

struct AttnTcParams {
  const __nv_bfloat16* x;    // block input, padded bf16 [B,18,18,192] (also the residual)
  __nv_bfloat16* out;        // x + proj(attention(qkv(norm(x)))), padded bf16 [B,18,18,192], halo written
  const uint8_t* wpack;      // attn_tc_pack_weights image (device)
  const float* bias_qkv;     // attn.qkv.bias [576]
  const float* bias_proj;    // attn.proj.bias [192]
  const float* gamma;        // attn.norm.weight [192]
  const float* beta;         // attn.norm.bias [192]
  int B;
  float* dbg;               // tests only (or null): intermediates of image 0, see ATTN_DBG_* offsets
};

// debug dump layout (floats): normalised input [256][192] | q,k,v + bias [256][576] | attention output y [256][192] |
// softmax denominators [256][4]
constexpr size_t ATTN_DBG_XN = 0, ATTN_DBG_QKV = 256 * 192, ATTN_DBG_Y = ATTN_DBG_QKV + 256 * 576,
                 ATTN_DBG_L = ATTN_DBG_Y + 256 * 192, ATTN_DBG_FLOATS = ATTN_DBG_L + 256 * 4;

size_t attn_tc_wpack_bytes();
// qkv_w [576][192], proj_w [192][192] (PyTorch [out][in] of the 1x1 convs) -> the shared-memory images the kernel
// bulk-copies: per head [3 K blocks of 64 channels][144 rows = q|k|v of the head][128 B, SWIZZLE_128B], then the
// projection [3][192][128 B]
void attn_tc_pack_weights(const float* qkv_w, const float* proj_w, uint8_t* out_host);
int launch_attn_block_tc(const AttnTcParams& p, int sm_count, cudaStream_t st);

}  // namespace tcs
