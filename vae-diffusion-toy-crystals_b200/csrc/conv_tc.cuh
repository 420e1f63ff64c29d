// conv_tc.cuh — host interface of the tcgen05 implicit-GEMM convolution (conv_tc.cu).
#pragma once
#include <vector>

#include "common.cuh"

namespace tcs {

struct ConvTcParams {
  int n_mtiles, n_ntiles;   // tiles = n_mtiles * n_ntiles
  int tiles_per_img;        // M tiles per image
  int H, W;                 // output spatial size
  int Rt;                   // image rows per 128-pixel sub-tile (= 128 / W)
  int T, KYG, KW;           // taps per stage, ky groups, kx count
  int stride, WR;           // conv stride; window rows per stage
  int nsrc, cblk[6], base_off[6];   // PHYSICAL sources (K segments): 1-2 normally, 3 per logical source in bf16x3 mode
  int msel[6];              // tensor map (0..3) each physical source reads
  int ctail[6];             // 1 = the source's last 64-channel block holds 32 channels only (two K steps instead of four)
  int ntot;                 // total output channels
  int kstages;              // pipeline stages (K iterations) per tile
  int b_rows;               // 512-byte rows of packed weights per stage and CTA
  int nstage;               // smem ring depth
  uint32_t a_bytes, stage_bytes;
  int pair;                 // EPI_EPS: 1 = the two sub-tiles are the same pixels of images 2i (cond) and 2i+1 (uncond)
  int kxn;                  // EPI_EPS: 1 = kx taps live in accumulator columns 0..2 (ConvGeom::kx_in_n)
  float guidance;           // EPI_EPS with pair: eps = e_u + guidance (e_c - e_u)
  double gn_inv_cnt;        // EPI_GN_FUSED: 1 / (H * W * channels per group)
  // geo = 1 ("tap-shift" geometry, 3x3 stride-1 layers): a 128-row sub-tile is 16 image rows x 8 pixels, the A operand
  // of a 64-channel block is ONE (16 + 2) x (8 MSUB + 2) pixel window in its own ring, and the nine taps are descriptor
  // start shifts into it; the weights stream through a second ring in stages of `tb` taps
  int geo;
  int P;                    // geo 1: window pixels per row (8 MSUB + 2); one window row = P * 128 B = the descriptor's SBO
  int tiles_x;              // geo 1: CTA tiles per image row
  int a_stages, tb;         // geo 1: A ring depth; taps per weight stage (3 or 1)
  uint32_t a_load_bytes;    // geo 1: bytes one window load delivers (a_bytes is its 1024-byte-aligned slot size)
  int ups;                  // 1 = fused bilinear x2 upsample (ConvGeom::ups): low-resolution windows in a ring of l_stages slots
  int l_stages;
  uint32_t l_bytes, l_load_bytes;
  int debug;                // TCS_DEBUG bits: 4 = per-lane stores instead of TMA stores (the reference of the TMA epilogues)
  EpiArgs epi;
};

struct ConvTcPlan {
  CUtensorMap mapA[4];   // [source] or, in bf16x3 mode, [hi0, lo0, hi1, lo1]
  CUtensorMap mapW;
  CUtensorMap mapO;   // EPI_PADDED / EPI_GN_FUSED: padded bf16 output, TMA-stored in 32-pixel x 32-channel boxes
  CUtensorMap mapO1;  // geo 1: the same tensor with a one-image-row box (the wrapped copies of rows 0 and H - 1)
  int geo = 0;
  int ups = 0;
  ConvTcParams p;
  int N;       // N tile (96 or 192)
  int epi;     // Epilogue
  int msub;    // 128-row sub-tiles per CTA tile
  int cg;      // 1 = one CTA per MMA, 2 = CTA pairs (tcgen05 cta_group::2, weights split across the pair)
  int grid;
  int cin[2] = {0, 0};       // channels of the logical sources
  int max_ctas = 0;          // CTAs of this kernel the device holds at once (cudaOccupancyMaxActiveClusters x 2 for pairs)
  bool coop_cluster = false; // launch the fused-GroupNorm CTA pairs with the cooperative attribute as well
  size_t smem;
  bool valid = false;
};

// number of K stages and packed weight element count for a geometry
int conv_tc_kstages(const ConvGeom& g);
size_t conv_tc_packed_elems(const ConvGeom& g);
// weight [ntot][cin_total][k][k] fp32 (PyTorch layout) -> bf16 [kstage][N tile][CTA][tap][rows][64] (see conv_tc.cu)
// (bf16x3 mode: per logical source the K segments [w_hi, w_lo, w_hi], matching the A segments [a_hi, a_hi, a_lo])
void conv_tc_pack_weights(const ConvGeom& g, int epi, const float* w, __nv_bfloat16* out_host);
void conv_tc_tile_shape(const ConvGeom& g, int epi, int* N, int* cg);

// src0/src1: bf16 NHWC device tensors (padded or plain as g.in_pad says); wpacked: device bf16
// bf16x3 mode (g.split3): every fp32 source arrives as two bf16 tensors hi = bf16(a), lo = bf16(a - hi); src0/src1 are
// the hi parts, lo0/lo1 the lo parts.
int conv_tc_make_plan(ConvTcPlan* plan, const ConvGeom& g, const void* src0, const void* src1,
                      const __nv_bfloat16* wpacked, int epi, const EpiArgs& ea, int sm_count,
                      const void* lo0 = nullptr, const void* lo1 = nullptr);
int conv_tc_launch(const ConvTcPlan& plan, cudaStream_t stream);
int conv_tc_make_pair(ConvTcPlan* plan, const void* src, int B);
// grid for B images (persistent: <= one CTA per SM; whole image groups for EPI_GN_FUSED)
int conv_tc_grid(const ConvTcPlan& plan, int B, int sm_count);

}  // namespace tcs
