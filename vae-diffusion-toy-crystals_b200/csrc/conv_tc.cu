// conv_tc.cu — circular-padded convolution as an implicit GEMM on the 5th-gen tensor cores.
//
// Replaces every nn.Conv2d(padding_mode="circular") of CondUNetTiny except the 1-channel
// input conv and the 1-channel output conv (reference: src/toycrystals/models/sde_score_model.py
// :102,105 (_ConvBlock), :208,210 (ds1/ds2), :133-134 (attn qkv/proj), :218,222 (us*_conv)).
//
//   D[M = B*H*W pixels, N = C_out] = sum over (source, 32-channel block, kx, ky)  A_tap[M,32] * W_tap[N,32]^T
//
// * activations are bf16 NHWC with a 1-pixel circular halo, so every tap is a plain TMA box;
// * one pipeline stage = one (source, 32-ch block, kx[, ky parity]) "window": the TMA box holds
//   Rt*MSUB + T - 1 image rows of the tile's full width, and the T taps that differ only in ky
//   are row-shifted views of it (shift = W*64 B, a multiple of the 512 B swizzle period), so A
//   is fetched T times less often than tap-by-tap;
// * operands sit in shared memory in the K-major SWIZZLE_64B canonical layout (one 64 B row
//   per pixel / per output channel), accumulators in TMEM (fp32), double buffered;
// * warp 0 = TMA producer, warps 1 and 18 = tcgen05.mma issuers (one elected lane each), warps 2..17 = epilogue in two
//   groups of 8, one per TMEM accumulator set (tcgen05.ld -> bias / GroupNorm + SiLU / halo writes via TMA stores);
// * CTA pairs (cluster of 2, cta_group::2): the weight tile is split across the two CTAs' shared memory;
// * persistent grid: one CTA per SM looping over M tiles.
#include "conv_tc.cuh"
#include "tc_ptx.cuh"

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <type_traits>
#include <vector>

// -DTCS_KERNEL_PROFILE=1 compiles the in-kernel clock64 phase profiler in (printed per layer with TCS_DEBUG=128);
// the default build leaves it out so that it costs no registers
#ifndef TCS_KERNEL_PROFILE
#define TCS_KERNEL_PROFILE 0
#endif

namespace tcs {


constexpr int EPI_WARPS = 16;          // two groups of 8: group g owns TMEM accumulator set g, i.e. every second tile
constexpr int GRP_WARPS = EPI_WARPS / 2;
constexpr int UC = 96;                 // accumulator columns per epilogue warp (4 lane quarters x 2 column units cover 192)
constexpr int BLK = 32;                // channels per staged output block (three blocks per warp and tile)
constexpr int TC_THREADS = 64 + 32 * EPI_WARPS + 32;   // + a second MMA-issuing warp for the MSUB = 2 tiles
// UPS kernels: warps 19..22 blend the upsampled windows (two more padding warps, so that none of them shares a scheduler
// with the MMA-issuing warps 1 and 18, cost more than they gain: 800 threads leave 72 registers per thread)
constexpr int UPS_EXTRA_THREADS = 4 * 32;
constexpr int MAX_STAGES = 12;
constexpr int MAX_A_STAGES = 4;
// K block of a pipeline stage: 64 input channels = one 128-byte row per pixel / per output channel (SWIZZLE_128B).
// 128-byte rows instead of 64-byte ones halve the number of TMA / L2 requests per operand byte, which is what bounds the
// operand feed (round 2: moving the weights from 64-byte to 512-byte rows alone was worth +8 %).  A source whose channel
// count is not a multiple of 64 (96 = 64 + 32) ends in a half block: TMA zero-fills the missing channels without
// requesting them and the issuer skips their two K steps.
constexpr int KB = 64;
constexpr uint32_t ROWB = KB * 2;
constexpr int SLAB_BUFS = 2;                            // staging blocks per epilogue warp (1 frees an operand stage: measured no gain)
constexpr uint32_t EPI_WARP_SLAB = SLAB_BUFS * 32 * BLK * 2;    // per epilogue warp: 32 px x BLK ch bf16 blocks
constexpr uint32_t EPI_SLAB_BYTES = EPI_WARPS * EPI_WARP_SLAB;
constexpr uint32_t EPI_BIAS_BYTES = 576 * 4;
// shared memory a CTA may use: 227 KB minus the static part (barriers) and the worst-case 1024-byte alignment of the ring
constexpr size_t TC_SMEM_MAX = 227 * 1024 - 512;
__host__ __device__ constexpr uint32_t bias_bytes_of(int ntot) { return (static_cast<uint32_t>(ntot) * 4u + 127u) & ~127u; }
struct EpiGroupSmem {          // per epilogue warp group (EPI_GN_FUSED)
  float scale[192], shift[192];
  float red[GRP_WARPS][16];    // per warp: (sum, sum of squares) of the 8 GroupNorm groups over its block
  float mean[8], rstd[8];
};
struct EpiFusedSmem {          // EPI_GN_FUSED scratch (lives right after the bias)
  float gamma[192], beta[192];
  EpiGroupSmem grp[2];
};
constexpr uint32_t EPI_FUSED_BYTES = sizeof(EpiFusedSmem);
// The G CTAs of an image wait for each other's GroupNorm partial sums (one L2 round trip when they run in lock step).
// Co-residency of the whole grid is guaranteed by the launch (cooperative attribute, grid clamped to
// cudaOccupancyMaxActiveClusters), so this bound only turns a protocol bug into a launch failure instead of a hang.
// (TCS_EXCHANGE_TIMEOUT=<cycles> overrides it: instrumented ncu passes run the kernel orders of magnitude slower.)
constexpr long long EXCHANGE_TIMEOUT_CYCLES = 1000000000LL;   // ~0.5 s

__device__ __forceinline__ void st_relaxed_gpu_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.relaxed.gpu.global.b64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_relaxed_gpu_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.b64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void epi_bar_sync(int grp) { asm volatile("bar.sync %0, %1;" ::"r"(1 + grp), "n"(32 * GRP_WARPS) : "memory"); }
// fp16 pair (a in the low half), saturating to the largest finite value
__device__ __forceinline__ uint32_t pack_f16x2_sat(float a, float b) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}
__device__ __forceinline__ float2 unpack_f16x2(uint32_t v) {
  return __half22float2(*reinterpret_cast<const __half2*>(&v));
}
__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&h);
}
// SiLU(y) = y * sigmoid(y) = h + h * tanh(h), h = y/2: one MUFU instead of two (ex2 + rcp)
__device__ __forceinline__ float silu_fast(float y) {
  const float h = 0.5f * y;
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
  return fmaf(h, t, h);
}
__device__ __forceinline__ void store_with_halo(__nv_bfloat16* obase, size_t pix, int wy, int wx, int Wp, int ldo,
                                                int ch, const uint32_t* pk);

// packed fp32x2 arithmetic (sm_100: FFMA2 / FADD2): halves the epilogue's floating-point instruction count
__device__ __forceinline__ void fma2(float& d0, float& d1, float a0, float a1, float b0, float b1, float c0, float c1) {
  asm("{\n\t.reg .b64 ra, rb, rc, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmov.b64 rc, {%6, %7};\n\t"
      "fma.rn.f32x2 rd, ra, rb, rc;\n\tmov.b64 {%0, %1}, rd;\n\t}"
      : "=f"(d0), "=f"(d1) : "f"(a0), "f"(a1), "f"(b0), "f"(b1), "f"(c0), "f"(c1));
}
__device__ __forceinline__ void add2(float& d0, float& d1, float a0, float a1, float b0, float b1) {
  asm("{\n\t.reg .b64 ra, rb, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\t"
      "add.rn.f32x2 rd, ra, rb;\n\tmov.b64 {%0, %1}, rd;\n\t}"
      : "=f"(d0), "=f"(d1) : "f"(a0), "f"(a1), "f"(b0), "f"(b1));
}
__device__ __forceinline__ float tanh_fast(float x) {
#ifdef TCS_NO_TANH
  return x * 0.25f;   // timing experiment only: no MUFU in the fused epilogue
#else
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(x));
  return t;
#endif
}
__device__ __forceinline__ void st_shared_u4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void ld_shared_u4(uint32_t addr, uint32_t& a, uint32_t& b, uint32_t& c, uint32_t& d) {
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "r"(addr) : "memory");
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, uint32_t src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(map)), "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
// 32 pixels (one per lane, consecutive in an image row) x 32 bf16 channels -> padded NHWC output.
// W >= 32: the warp stages the 2 KB block in a SWIZZLE_64B slab (two halves, double buffered) and one lane TMA-stores it
// (plus the wrapped row copy); only the lanes on the left/right image border write their column-halo copy themselves.
// W == 16: plain per-lane 16-byte stores (the 16x16 layers are small).
// GEO == 1: the 32 lanes are 4 image rows x 8 pixels (lane = 8 * row + pixel); one TMA store of an 8-pixel x 4-row box,
// plus a one-row box (mapO1, geo_H = image height) when the block holds image row 0 or H - 1 (the wrapped halo rows).
template <int GEO = 0, int SB = SLAB_BUFS>
__device__ __forceinline__ void store_padded_block(const CUtensorMap* mapO, bool use_tma, uint32_t slab, uint32_t& slab_buf,
                                                   int lane, __nv_bfloat16* obase, size_t pix, int wy, int wx, int Wp,
                                                   int ldo, int ch, int img, int y, int x, const uint32_t* pk,
                                                   long long* tacc = nullptr, int h16 = 0,
                                                   const CUtensorMap* mapO1 = nullptr, int geo_H = 0) {
  if (!use_tma) {
    store_with_halo(obase, pix, wy, wx, Wp, ldo, ch, pk);
    return;
  }
  long long c0 = tacc ? clock64() : 0;
  if (lane == 0) ptx::bulk_wait_read<SB - 1>();   // the staging block about to be overwritten has been read
  __syncwarp();
  if (tacc) { const long long c1 = clock64(); tacc[0] += c1 - c0; c0 = c1; }
  const uint32_t base = slab + (SB == 2 ? slab_buf * 2048 : 0);
  const uint32_t dst = base + lane * 64;
  const int sw = (lane >> 1) & 3;
#pragma unroll
  for (int j = 0; j < 4; ++j) st_shared_u4(dst + ((j ^ sw) << 4), pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
  ptx::fence_proxy_async();
  __syncwarp();
  if (tacc) { const long long c1 = clock64(); tacc[1] += c1 - c0; c0 = c1; }
  if (lane == 0) {   // lane 0 holds the first pixel of the block: (y, x) -> padded (y+1, x+1)
    if (GEO == 1) {
      tma_store_4d(mapO, base, ch, x + 1, y + 1, img);
      if (y == 0) tma_store_4d(mapO1, base, ch, x + 1, geo_H + 1, img);                  // row 0 -> also padded row H + 1
      if (y + 4 == geo_H) tma_store_4d(mapO1, base + 3 * 512, ch, x + 1, 0, img);        // row H - 1 -> also padded row 0
    } else if (h16 == 0) {
      tma_store_4d(mapO, base, ch, x + 1, y + 1, img);
      if (wy) tma_store_4d(mapO, base, ch, x + 1, y + 1 + wy, img);
    } else {         // 16-pixel rows: the block is image rows y (lanes 0-15) and y + 1 (lanes 16-31), one 16-pixel box each
      tma_store_4d(mapO, base, ch, 1, y + 1, img);
      tma_store_4d(mapO, base + 1024, ch, 1, y + 2, img);
      if (y == 0) tma_store_4d(mapO, base, ch, 1, h16 + 1, img);                 // row 0 -> also padded row H + 1
      if (y + 1 == h16 - 1) tma_store_4d(mapO, base + 1024, ch, 1, 0, img);      // row H - 1 -> also padded row 0
    }
    ptx::bulk_commit();
  }
  __syncwarp();
  if (tacc) { const long long c1 = clock64(); tacc[2] += c1 - c0; c0 = c1; }
  slab_buf ^= 1;
  if (wx) {   // column halo (and the corner when this pixel is also on a border row)
    uint4* d0 = reinterpret_cast<uint4*>(obase + (pix + wx) * ldo + ch);
#pragma unroll
    for (int i = 0; i < 4; ++i) d0[i] = make_uint4(pk[4 * i], pk[4 * i + 1], pk[4 * i + 2], pk[4 * i + 3]);
    if (wy) {
      uint4* d1 = reinterpret_cast<uint4*>(obase + (pix + static_cast<long long>(wy) * Wp + wx) * ldo + ch);
#pragma unroll
      for (int i = 0; i < 4; ++i) d1[i] = make_uint4(pk[4 * i], pk[4 * i + 1], pk[4 * i + 2], pk[4 * i + 3]);
    }
  }
}

// BLK bf16 channels of one pixel -> padded NHWC tensor, duplicated onto the circular halo where needed
__device__ __forceinline__ void store_with_halo(__nv_bfloat16* obase, size_t pix, int wy, int wx, int Wp, int ldo,
                                                int ch, const uint32_t* pk) {
#pragma unroll
  for (int cy = 0; cy < 2; ++cy) {
    if (cy == 1 && wy == 0) continue;
#pragma unroll
    for (int cx = 0; cx < 2; ++cx) {
      if (cx == 1 && wx == 0) continue;
      const size_t dp = pix + static_cast<long long>(cy ? wy : 0) * Wp + (cx ? wx : 0);
      uint4* dst = reinterpret_cast<uint4*>(obase + dp * ldo + ch);
#pragma unroll
      for (int i = 0; i < BLK / 8; ++i) dst[i] = make_uint4(pk[4 * i], pk[4 * i + 1], pk[4 * i + 2], pk[4 * i + 3]);
    }
  }
}

// tile index -> (M tile, N tile).  With CTA pairs the two CTAs of a pair (consecutive tile indices) must share the
// N tile, because one MMA reads the weight tile half from each of them.
template <int CG>
__device__ __forceinline__ void tile_to_mn(int tile, int n_ntiles, int& mt, int& nt) {
  if (CG == 2) {
    const int pt = tile >> 1;
    nt = pt % n_ntiles;
    mt = ((pt / n_ntiles) << 1) | (tile & 1);
  } else {
    mt = tile / n_ntiles;
    nt = tile - mt * n_ntiles;
  }
}

struct __align__(8) TcBarriers {
  uint64_t full[MAX_STAGES];
  uint64_t empty[MAX_STAGES];
  uint64_t fullA[MAX_A_STAGES];    // geo 1: the window ring
  uint64_t emptyA[MAX_A_STAGES];
  uint64_t fullL[2];               // UPS: the low-resolution window ring
  uint64_t emptyL[2];
  uint64_t tmem_full[2];
  uint64_t tmem_empty[2];
  uint32_t tmem_base;
};

// CG = 2: the kernel runs as CTA pairs (cluster of 2).  Each CTA still owns its own M tile (its 128-row sub-tiles,
// its TMEM accumulators, its epilogue), but one tcgen05.mma.cta_group::2 of the leader drives both tensor cores
// with M = 256 and reads the weight tile HALF from each CTA's shared memory: every CTA fetches only N/2 weight
// rows per stage, which halves the dominant L2 -> SM operand stream.
//
// GEO = 1 (the 3x3 stride-1 layers, ~90 % of the FLOPs): "tap-shift" geometry.  A 128-row sub-tile is 16 image rows x 8
// pixels, so that an 8-row core group of the UMMA descriptor is 8 consecutive pixels of ONE image row and the group
// stride (SBO) is one row of the shared-memory window.  The window of a 64-channel block, (16 + 2) x (8 MSUB + 2) pixels
// with the halo, is loaded ONCE and all nine taps are start-address shifts of (ky P + kx) * 128 B into it (the swizzle
// is a function of the absolute shared-memory address, so neither the 128-byte shifts nor a window pitch that is not a
// multiple of 1024 B need the descriptor's base-offset field: probed on the hardware by tools/umma_shift_test.cu).
// GEO = 0 fetched a full-width window per kx (each input pixel 4.5 x per tile); GEO = 1 fetches it 1.27 x (MSUB = 2),
// which halves the L2 -> SM operand stream that bounded the 64x64 layers (no-TMA experiment: +39 %).  The windows have
// their own ring (fullA / emptyA); the weights stream through the stage ring in stages of p.tb taps.
// UPS = 1 (us1_conv / us2_conv): the source is the HALF-resolution padded tensor and nn.Upsample(scale_factor=2,
// mode="bilinear") (sde_score_model.py:217,221) happens on the way into shared memory: the TMA producer loads the
// (8 + 2) x (4 MSUB + 2) low-resolution window of a 64-channel block into a ring of its own, four extra warps
// (19..22) blend it into the (16 + 2) x (8 MSUB + 2) tap-shift window (edge clamp of the upsample, circular wrap of the
// conv: the first / last window rows and columns of border tiles are plain copies) and arrive on the window's barrier.
// The upsampled tensor never exists in memory (it was 4x the size of the input, written and read back once per pass).
template <int N, int EPI, int MSUB, int CG, int GEO, int UPS = 0>
__global__ void __launch_bounds__(TC_THREADS + UPS_EXTRA_THREADS * UPS, 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap mapA0, const __grid_constant__ CUtensorMap mapA1,
               const __grid_constant__ CUtensorMap mapA2, const __grid_constant__ CUtensorMap mapA3,
               const __grid_constant__ CUtensorMap mapW, const __grid_constant__ CUtensorMap mapO,
               const __grid_constant__ CUtensorMap mapO1, const ConvTcParams p) {
  static_assert(GEO == 0 || (EPI != EPI_EPS && EPI != EPI_PLAIN), "tap-shift geometry: padded / fp32 outputs only");
  static_assert(UPS == 0 || (GEO == 1 && CG == 2 && EPI == EPI_PADDED), "fused upsample: tap-shift CTA pairs, padded output");
  constexpr int ACC_STRIDE = (N * MSUB <= 128) ? 128 : 256;  // TMEM columns per accumulator stage
  static_assert(N * MSUB <= 256, "accumulator does not fit a double-buffered TMEM stage");

  extern __shared__ uint8_t smem_raw[];
  __shared__ TcBarriers bars;

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);   // warp-uniform for the compiler (uniform datapath)
  const int lane = threadIdx.x & 31;
  const uint32_t smem_base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  const int n_tiles = p.n_mtiles * p.n_ntiles;
  // after the operand ring: 16 epilogue warps x 2 x 2 KB staging blocks (fp16 stash of the fused epilogue, TMA-store
  // source of every bf16 output), then the bias
  const uint32_t l_ring = smem_base + (GEO == 1 ? p.a_stages * p.a_bytes : 0u);   // UPS: low-resolution windows after the window ring
  const uint32_t b_ring = l_ring + (UPS ? p.l_stages * p.l_bytes : 0u);           // geo 1: windows first, then weight stages
  const uint32_t slab_base = b_ring + p.nstage * p.stage_bytes;
  // UPS kernels stage their outputs in ONE 2 KB block per epilogue warp (measured neutral for the epilogue) and spend the
  // 32 KB on a third window stage (us1_conv) or a third weight stage (us2_conv)
  constexpr int SB = UPS ? 1 : SLAB_BUFS;
  constexpr uint32_t WARP_SLAB = SB * 32 * BLK * 2, SLAB_BYTES = EPI_WARPS * WARP_SLAB;
  float* bias_s = reinterpret_cast<float*>(smem_raw + (slab_base - ptx::smem_u32(smem_raw)) + SLAB_BYTES);
  for (int i = threadIdx.x; i < p.ntot; i += blockDim.x) {
    float b = p.epi.bias[i];
    if constexpr (EPI == EPI_GN_FUSED) {
      // GroupNorm is shift invariant: the fused epilogue works on v + bias - K_g with K_g = the mean of the group's
      // biases, so that a bias far from zero (trained weights: |mean| >> std of the group) costs neither fp16 stash bits
      // (rounding 2^-11 |v + bias - K_g| instead of 2^-11 |v + bias|) nor the cancellation of E[v^2] - mean^2
      constexpr int CPGN = N / 8;
      const int g0 = i - i % CPGN;
      float k = 0.f;
#pragma unroll
      for (int j = 0; j < CPGN; ++j) k += p.epi.bias[g0 + j];
      b -= k * (1.0f / CPGN);
    }
    bias_s[i] = b;
  }
  EpiFusedSmem* fs = reinterpret_cast<EpiFusedSmem*>(reinterpret_cast<uint8_t*>(bias_s) + (GEO == 1 ? bias_bytes_of(p.ntot) : EPI_BIAS_BYTES));
  if constexpr (EPI == EPI_GN_FUSED)
    for (int i = threadIdx.x; i < N; i += blockDim.x) { fs->gamma[i] = p.epi.gamma[i]; fs->beta[i] = p.epi.beta[i]; }

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&mapA0);
    ptx::prefetch_tmap(&mapA1);
    if (p.nsrc > 2) { ptx::prefetch_tmap(&mapA2); ptx::prefetch_tmap(&mapA3); }
    ptx::prefetch_tmap(&mapW);
    if (EPI != EPI_EPS) ptx::prefetch_tmap(&mapO);
    if (GEO == 1) ptx::prefetch_tmap(&mapO1);
    for (int s = 0; s < p.nstage; ++s) {
      ptx::mbar_init(ptx::smem_u32(&bars.full[s]), 1);
      ptx::mbar_init(ptx::smem_u32(&bars.empty[s]), p.issuers);     // one tcgen05.commit per issuing thread
    }
    if (GEO == 1)
      for (int s = 0; s < p.a_stages; ++s) {
        ptx::mbar_init(ptx::smem_u32(&bars.fullA[s]), UPS ? 4 * CG : 1);   // UPS: one arrival per blending warp of the pair
        ptx::mbar_init(ptx::smem_u32(&bars.emptyA[s]), p.issuers);
      }
    if (UPS)
      for (int s = 0; s < p.l_stages; ++s) {
        ptx::mbar_init(ptx::smem_u32(&bars.fullL[s]), 1);
        ptx::mbar_init(ptx::smem_u32(&bars.emptyL[s]), 4);
      }
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(ptx::smem_u32(&bars.tmem_full[a]), p.issuers);
      ptx::mbar_init(ptx::smem_u32(&bars.tmem_empty[a]), GRP_WARPS * CG);
    }
    ptx::fence_barrier_init();
  }
  const uint32_t cta_rank = (CG == 2) ? ptx::cluster_ctarank() : 0u;
  constexpr int NB = N / CG;    // weight rows this CTA keeps per tap
  if (warp == 1) {
    if (CG == 2) ptx::tmem_alloc_512_2sm(ptx::smem_u32(&bars.tmem_base));
    else ptx::tmem_alloc_512(ptx::smem_u32(&bars.tmem_base));
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (CG == 2) ptx::cluster_sync_all();   // peer barriers are initialised before anyone signals them
  ptx::tc_fence_after();
  const uint32_t tmem_base = bars.tmem_base;

  if (warp == 0 && GEO == 1) {
    // ============================== TMA producer, tap-shift geometry ==========
    uint32_t sa = 0, pa = 0, sb = 0, pb = 0;
    const int b_stages_per_kx = 3 / p.tb;
    const int b_rows_full = 3 * NB / 4;          // 512-byte rows of the three ky taps of one (block, kx) in the packed weights
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      int mt, nt;
      tile_to_mn<CG>(tile, p.n_ntiles, mt, nt);
      const int b = mt / p.tiles_per_img, t = mt - b * p.tiles_per_img;
      const int ty = t / p.tiles_x, tx = t - ty * p.tiles_x;
      int ks = 0;
      for (int src = 0; src < p.nsrc; ++src) {
        const int ms = p.msel[src];
        const CUtensorMap* mapA = ms == 0 ? &mapA0 : (ms == 1 ? &mapA1 : (ms == 2 ? &mapA2 : &mapA3));
        for (int cb = 0; cb < p.cblk[src]; ++cb) {
          if constexpr (UPS) {   // low-resolution window -> its own ring (this CTA's barrier); warps 19..22 fill the A ring
            // The window of the NEXT block is requested before this block's weights: the weight ring blocks this warp until
            // the MMAs make progress, and a window that is only requested then arrives (and is blended) too late.
            auto issue_low = [&](int tl, int cbx) {
              int mt2, nt2;
              tile_to_mn<CG>(tl, p.n_ntiles, mt2, nt2);
              const int b2 = mt2 / p.tiles_per_img, t2 = mt2 - b2 * p.tiles_per_img;
              const int ty2 = t2 / p.tiles_x, tx2 = t2 - ty2 * p.tiles_x;
              ptx::mbar_wait(ptx::smem_u32(&bars.emptyL[sa]), pa ^ 1);
              if (lane == 0) {
                const uint32_t full = ptx::smem_u32(&bars.fullL[sa]);
                ptx::mbar_expect_tx(full, p.l_load_bytes);
                ptx::tma_load_4d(l_ring + sa * p.l_bytes, mapA, full, cbx * KB, tx2 * 4 * MSUB + p.base_off[0], ty2 * 8 + p.base_off[0], b2);
              }
              __syncwarp();
              if (++sa == static_cast<uint32_t>(p.l_stages)) { sa = 0; pa ^= 1; }
            };
            if (tile == static_cast<int>(blockIdx.x) && cb == 0) issue_low(tile, 0);
            int ntile = tile, ncb = cb + 1;
            if (ncb == p.cblk[0]) { ncb = 0; ntile = tile + static_cast<int>(gridDim.x); }
            if (ntile < n_tiles) issue_low(ntile, ncb);
          } else {
          ptx::mbar_wait(ptx::smem_u32(&bars.emptyA[sa]), pa ^ 1);
          const bool stale = (p.debug & 8) && (pa || tile != static_cast<int>(blockIdx.x));   // experiment: no TMA
          if (lane == 0) {
            const uint32_t full = ptx::smem_u32(&bars.fullA[sa]);
            const uint32_t a_dst = smem_base + sa * p.a_bytes;
            if (stale) {
              if (CG == 1 || cta_rank == 0) ptx::mbar_arrive(full);
            } else if (CG == 2) {
              if (cta_rank == 0) ptx::mbar_expect_tx(full, 2 * p.a_load_bytes);
              ptx::tma_load_4d_2sm(a_dst, mapA, full, cb * KB, tx * 8 * MSUB + p.base_off[src], ty * 16 + p.base_off[src], b);
            } else {
              ptx::mbar_expect_tx(full, p.a_load_bytes);
              ptx::tma_load_4d(a_dst, mapA, full, cb * KB, tx * 8 * MSUB + p.base_off[src], ty * 16 + p.base_off[src], b);
            }
          }
          __syncwarp();
          if (++sa == static_cast<uint32_t>(p.a_stages)) { sa = 0; pa ^= 1; }
          }
          for (int kx = 0; kx < 3; ++kx, ++ks)
            for (int jb = 0; jb < b_stages_per_kx; ++jb) {
              ptx::mbar_wait(ptx::smem_u32(&bars.empty[sb]), pb ^ 1);
              const bool stale_b = (p.debug & 8) && (pb || tile != static_cast<int>(blockIdx.x));
              if (lane == 0) {
                const uint32_t full = ptx::smem_u32(&bars.full[sb]);
                const uint32_t b_dst = b_ring + sb * p.stage_bytes;
                const int row0 = ((ks * p.n_ntiles + nt) * CG + static_cast<int>(cta_rank)) * b_rows_full + jb * p.b_rows;
                if (stale_b) {
                  if (CG == 1 || cta_rank == 0) ptx::mbar_arrive(full);
                } else if (CG == 2) {
                  if (cta_rank == 0) ptx::mbar_expect_tx(full, 2 * p.tb * NB * ROWB);
                  ptx::tma_load_2d_2sm(b_dst, &mapW, full, 0, row0);
                } else {
                  ptx::mbar_expect_tx(full, p.tb * NB * ROWB);
                  ptx::tma_load_2d(b_dst, &mapW, full, 0, row0);
                }
              }
              __syncwarp();
              if (++sb == static_cast<uint32_t>(p.nstage)) { sb = 0; pb ^= 1; }
            }
        }
      }
    }
  } else if (warp == 0) {
    // ============================== TMA producer ==============================
    uint32_t stage = 0, phase = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      int mt, nt;
      tile_to_mn<CG>(tile, p.n_ntiles, mt, nt);
      // pair mode (EPI_EPS + CFG): tile = the same Rt rows of images 2i and 2i+1, one window each
      const int rows_per_tile = p.pair ? p.Rt : p.Rt * MSUB;
      const int b = (mt / p.tiles_per_img) * (p.pair ? 2 : 1);
      const int y0 = (mt % p.tiles_per_img) * rows_per_tile;
      int ks = 0;
      for (int src = 0; src < p.nsrc; ++src) {
        const int ms = p.msel[src];
        const CUtensorMap* mapA = ms == 0 ? &mapA0 : (ms == 1 ? &mapA1 : (ms == 2 ? &mapA2 : &mapA3));
        for (int cb = 0; cb < p.cblk[src]; ++cb)
          for (int kyg = 0; kyg < p.KYG; ++kyg)
            for (int kx = 0; kx < p.KW; ++kx, ++ks) {
              ptx::mbar_wait(ptx::smem_u32(&bars.empty[stage]), phase ^ 1);
              if ((p.debug & 8) && (phase || tile != static_cast<int>(blockIdx.x))) {   // experiment: stale operands, no TMA
                if (lane == 0 && (CG == 1 || cta_rank == 0)) ptx::mbar_arrive(ptx::smem_u32(&bars.full[stage]));
                __syncwarp();
                if (++stage == static_cast<uint32_t>(p.nstage)) { stage = 0; phase ^= 1; }
                continue;
              }
              if (lane == 0) {
                const uint32_t full = ptx::smem_u32(&bars.full[stage]);
                const uint32_t a_dst = smem_base + stage * p.stage_bytes;
                const uint32_t b_dst = a_dst + p.a_bytes;
                if (CG == 2) {
                  // both CTAs' loads complete on the LEADER's full barrier; the leader arms it for both
                  if (cta_rank == 0) ptx::mbar_expect_tx(full, 2 * (p.a_bytes + p.T * NB * ROWB));
                  ptx::tma_load_4d_2sm(a_dst, mapA, full, cb * KB, kx + p.kxn + p.base_off[src],
                                       p.stride * y0 + kyg + p.base_off[src], b);
                  if (p.pair)
                    ptx::tma_load_4d_2sm(a_dst + p.a_bytes / 2, mapA, full, cb * KB, kx + p.kxn + p.base_off[src],
                                         p.stride * y0 + kyg + p.base_off[src], b + 1);
                  // weights: ONE box of 512-byte rows (the T taps of this CTA's N/2 rows, stored in global memory as the
                  // exact SWIZZLE_64B shared-memory image): 4x fewer TMA/L2 requests than 64-byte rows
                  ptx::tma_load_2d_2sm(b_dst, &mapW, full, 0,
                                       ((ks * p.n_ntiles + nt) * 2 + static_cast<int>(cta_rank)) * p.b_rows);
                } else {
                  ptx::mbar_expect_tx(full, p.a_bytes + p.T * N * ROWB);
                  ptx::tma_load_4d(a_dst, mapA, full, cb * KB, kx + p.kxn + p.base_off[src],
                                   p.stride * y0 + kyg + p.base_off[src], b);
                  if (p.pair)
                    ptx::tma_load_4d(a_dst + p.a_bytes / 2, mapA, full, cb * KB, kx + p.kxn + p.base_off[src],
                                     p.stride * y0 + kyg + p.base_off[src], b + 1);
                  ptx::tma_load_2d(b_dst, &mapW, full, 0, (ks * p.n_ntiles + nt) * p.b_rows);
                }
              }
              __syncwarp();
              if (++stage == static_cast<uint32_t>(p.nstage)) { stage = 0; phase ^= 1; }
            }
      }
    }
  } else if ((warp == 1 || (warp == 2 + EPI_WARPS && p.issuers == 2)) && cta_rank == 0) {
    // ============================== MMA issuer (leader CTA only when CG == 2) ====
    // The issue loop is the critical resource of this kernel: one thread needs ~60 cycles per tcgen05.mma (descriptor
    // arithmetic on the uniform datapath + the elect loop the compiler wraps around UTCHMMA), more than the 48 tensor
    // cycles an N = 96 MMA takes (measured: with the epilogue and the TMA loads switched off the N = 96 layers ran at
    // 770 TFLOP/s with one issuing thread and 990 with two).  With p.issuers == 2 the two 128-row sub-tiles of a tile
    // are issued by two warps (sub 0: warp 1, sub 1: warp 10); each commits its own MMAs, so the stage / accumulator
    // barriers expect two arrivals.  The sub-tile range and the tap count are compile-time in mma_role.
    constexpr uint32_t idesc = make_idesc(128 * CG, N);
    if constexpr (GEO == 1) {
      // ---- tap-shift geometry: per 64-channel block one window, nine taps = start shifts; weights in stages of p.tb taps
      auto run1 = [&](auto sub_lo_c, auto sub_hi_c) {
        constexpr int SUB_LO = decltype(sub_lo_c)::value, SUB_HI = decltype(sub_hi_c)::value;
        uint32_t sa = 0, pa = 0, sb = 0, pb = 0, acc = 0, acc_phase = 0;
        const int b_stages_per_kx = 3 / p.tb;
        const uint32_t ky_inc = static_cast<uint32_t>(p.P) * (ROWB >> 4);   // one window row, in 16-byte units
        int nblk = 0;
        for (int src = 0; src < p.nsrc; ++src) nblk += p.cblk[src];
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
          ptx::mbar_wait(ptx::smem_u32(&bars.tmem_empty[acc]), acc_phase ^ 1);
          ptx::tc_fence_after();
          const uint32_t d_tmem = tmem_base + acc * ACC_STRIDE;
          int blk = 0;
          for (int src = 0; src < p.nsrc; ++src)
            for (int cb = 0; cb < p.cblk[src]; ++cb, ++blk) {
              const int ksteps = (cb == p.cblk[src] - 1 && p.ctail[src]) ? 2 : 4;
              if (UPS) ptx::mbar_wait_cluster(ptx::smem_u32(&bars.fullA[sa]), pa);   // the peer's blending warps wrote its window
              else ptx::mbar_wait(ptx::smem_u32(&bars.fullA[sa]), pa);
              const uint64_t adesc = make_desc_sw128_sbo(smem_base + sa * p.a_bytes, static_cast<uint32_t>(p.P) * ROWB) +
                                     static_cast<uint64_t>(SUB_LO * 8 * (ROWB >> 4));
              for (int kx = 0; kx < 3; ++kx)
                for (int jb = 0; jb < b_stages_per_kx; ++jb) {
                  ptx::mbar_wait(ptx::smem_u32(&bars.full[sb]), pb);
                  ptx::tc_fence_after();
                  if (lane == 0) {
                    uint64_t bdj = make_desc_sw128(b_ring + sb * p.stage_bytes);
                    uint64_t adj = adesc + static_cast<uint64_t>(kx * (ROWB >> 4) + jb * p.tb * ky_inc);
                    for (int j = 0; j < p.tb; ++j) {
                      uint64_t ad = adj;
#pragma unroll
                      for (int sub = SUB_LO; sub < SUB_HI; ++sub) {
                        const uint32_t first = (blk | kx | jb | j) != 0 ? 1u : 0u;
                        if (CG == 2) {
                          ptx::umma_bf16_2sm(d_tmem + sub * N, ad, bdj, idesc, first);
                          ptx::umma_bf16_2sm(d_tmem + sub * N, ad + 2, bdj + 2, idesc, 1u);
                          if (ksteps == 4) {
                            ptx::umma_bf16_2sm(d_tmem + sub * N, ad + 4, bdj + 4, idesc, 1u);
                            ptx::umma_bf16_2sm(d_tmem + sub * N, ad + 6, bdj + 6, idesc, 1u);
                          }
                        } else {
                          ptx::umma_bf16(d_tmem + sub * N, ad, bdj, idesc, first);
                          ptx::umma_bf16(d_tmem + sub * N, ad + 2, bdj + 2, idesc, 1u);
                          if (ksteps == 4) {
                            ptx::umma_bf16(d_tmem + sub * N, ad + 4, bdj + 4, idesc, 1u);
                            ptx::umma_bf16(d_tmem + sub * N, ad + 6, bdj + 6, idesc, 1u);
                          }
                        }
                        ad += 8 * (ROWB >> 4);          // next sub-tile: 8 pixels to the right
                      }
                      adj += ky_inc;
                      bdj += (NB * ROWB) >> 4;
                    }
                    const bool last_of_blk = kx == 2 && jb == b_stages_per_kx - 1;
                    if (CG == 2) {
                      ptx::umma_commit_2sm(ptx::smem_u32(&bars.empty[sb]));
                      if (last_of_blk) ptx::umma_commit_2sm(ptx::smem_u32(&bars.emptyA[sa]));
                      if (last_of_blk && blk == nblk - 1) ptx::umma_commit_2sm(ptx::smem_u32(&bars.tmem_full[acc]));
                    } else {
                      ptx::umma_commit(ptx::smem_u32(&bars.empty[sb]));
                      if (last_of_blk) ptx::umma_commit(ptx::smem_u32(&bars.emptyA[sa]));
                      if (last_of_blk && blk == nblk - 1) ptx::umma_commit(ptx::smem_u32(&bars.tmem_full[acc]));
                    }
                  }
                  __syncwarp();
                  if (++sb == static_cast<uint32_t>(p.nstage)) { sb = 0; pb ^= 1; }
                }
              if (++sa == static_cast<uint32_t>(p.a_stages)) { sa = 0; pa ^= 1; }
            }
          if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
      };
      using J0 = std::integral_constant<int, 0>;
      using J1 = std::integral_constant<int, 1>;
      using JM = std::integral_constant<int, MSUB>;
      using JL = std::integral_constant<int, MSUB - 1>;
      if (p.issuers == 2) {
        if (warp == 1) run1(J0{}, J1{});
        else run1(JL{}, JM{});
      } else {
        run1(J0{}, JM{});
      }
    } else {
    const uint32_t row_shift = p.W * ROWB;  // one image row inside the window
    const uint32_t sub_stride = p.pair ? p.a_bytes / 2 : p.Rt * row_shift;  // second sub-tile: next window / next rows
    const uint32_t a_inc_j = row_shift >> 4, a_inc_sub = sub_stride >> 4;
    auto run = [&](auto sub_lo_c, auto sub_hi_c) {
      constexpr int SUB_LO = decltype(sub_lo_c)::value, SUB_HI = decltype(sub_hi_c)::value;
      uint32_t stage = 0, phase = 0, acc = 0, acc_phase = 0;
      const bool prof = TCS_KERNEL_PROFILE && (p.debug & 128) && blockIdx.x == 0 && warp == 1;
      long long w_empty = 0, w_full = 0, t_begin = prof ? clock64() : 0;
      int ntile = 0;
      const int stages_per_cb = p.KYG * p.KW;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        long long c0 = prof ? clock64() : 0;
        ptx::mbar_wait(ptx::smem_u32(&bars.tmem_empty[acc]), acc_phase ^ 1);
        ptx::tc_fence_after();
        if (prof) { w_empty += clock64() - c0; ++ntile; }
        int ks = 0;
        for (int src = 0; src < p.nsrc; ++src)
          for (int cb = 0; cb < p.cblk[src]; ++cb) {
            // K steps (16 channels each) of this channel block: 4, or 2 for the half block that ends a 96-channel source
            const int ksteps = (cb == p.cblk[src] - 1 && p.ctail[src]) ? 2 : 4;
            for (int sc = 0; sc < stages_per_cb; ++sc, ++ks) {
              c0 = prof ? clock64() : 0;
              ptx::mbar_wait(ptx::smem_u32(&bars.full[stage]), phase);
              ptx::tc_fence_after();
              if (prof) w_full += clock64() - c0;
              if (lane == 0) {
                // descriptors: one base per operand and stage, then 16-byte-unit increments
                const uint32_t a_base = smem_base + stage * p.stage_bytes;
                const uint64_t adesc = make_desc_sw128(a_base), bdesc = make_desc_sw128(a_base + p.a_bytes);
                const uint32_t d_tmem = tmem_base + acc * ACC_STRIDE;
                // running 64-bit descriptors: one uniform 64-bit add per operand and MMA (the issuing thread is the
                // bottleneck of this kernel, every instruction in this loop costs ~10 cycles of issue time per MMA)
                uint64_t adj = adesc + static_cast<uint64_t>(SUB_LO * a_inc_sub), bdj = bdesc;
                const uint64_t a_step = a_inc_j, a_sub = a_inc_sub;
                for (int j = 0; j < p.T; ++j) {
                  uint64_t ad = adj;
#pragma unroll
                  for (int sub = SUB_LO; sub < SUB_HI; ++sub) {
                    const uint32_t first = (ks | j) != 0 ? 1u : 0u;
                    if (CG == 2) {
                      ptx::umma_bf16_2sm(d_tmem + sub * N, ad, bdj, idesc, first);
                      ptx::umma_bf16_2sm(d_tmem + sub * N, ad + 2, bdj + 2, idesc, 1u);
                      if (ksteps == 4) {
                        ptx::umma_bf16_2sm(d_tmem + sub * N, ad + 4, bdj + 4, idesc, 1u);
                        ptx::umma_bf16_2sm(d_tmem + sub * N, ad + 6, bdj + 6, idesc, 1u);
                      }
                    } else {
                      ptx::umma_bf16(d_tmem + sub * N, ad, bdj, idesc, first);
                      ptx::umma_bf16(d_tmem + sub * N, ad + 2, bdj + 2, idesc, 1u);
                      if (ksteps == 4) {
                        ptx::umma_bf16(d_tmem + sub * N, ad + 4, bdj + 4, idesc, 1u);
                        ptx::umma_bf16(d_tmem + sub * N, ad + 6, bdj + 6, idesc, 1u);
                      }
                    }
                    ad += a_sub;
                  }
                  adj += a_step;
                  bdj += (NB * ROWB) >> 4;
                }
                if (CG == 2) {
                  ptx::umma_commit_2sm(ptx::smem_u32(&bars.empty[stage]));
                  if (ks == p.kstages - 1) ptx::umma_commit_2sm(ptx::smem_u32(&bars.tmem_full[acc]));
                } else {
                  ptx::umma_commit(ptx::smem_u32(&bars.empty[stage]));
                  if (ks == p.kstages - 1) ptx::umma_commit(ptx::smem_u32(&bars.tmem_full[acc]));
                }
              }
              __syncwarp();
              if (++stage == static_cast<uint32_t>(p.nstage)) { stage = 0; phase ^= 1; }
            }
          }
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
      if (prof && lane == 0)
        printf("[mma N=%d EPI=%d K=%d] tiles %d  cycles/tile %lld  wait tmem_empty %lld  wait full %lld\n", N, EPI, p.kstages, ntile,
               (clock64() - t_begin) / (ntile ? ntile : 1), w_empty / (ntile ? ntile : 1), w_full / (ntile ? ntile : 1));
    };
    using I0 = std::integral_constant<int, 0>;
    using I1 = std::integral_constant<int, 1>;
    using IM = std::integral_constant<int, MSUB>;
    using IL = std::integral_constant<int, MSUB - 1>;
    if (p.issuers == 2) {
      if (warp == 1) run(I0{}, I1{});
      else run(IL{}, IM{});
    } else {
      run(I0{}, IM{});
    }
    }
  } else if (UPS && warp >= 3 + EPI_WARPS) {
    // ============================== bilinear x2 into the window ring (UPS) ==============
    // thread = (16-byte channel chunk k, cell slot); a CELL is the 2 x 2 block of window pixels (2 cm + {0,1}, 2 cn + {0,1})
    // that blends the same four low-resolution pixels (cm + {0,1}, cn + {0,1}): rows / columns 2c and 2c + 1 weigh them
    // (3/4, 1/4) and (1/4, 3/4).  On a border tile the outermost cell row / column straddles the image edge: there the
    // upsample clamps and the conv wraps, and both are plain copies (weights (1, 0) and (0, 1)) because the low-resolution
    // halo already holds the wrapped pixel.  fp32 math, one rounding to bf16 (as the stand-alone upsample kernel did).
    if constexpr (UPS) {
      constexpr int P = 8 * MSUB + 2, CW = P / 2, LP = CW + 1;
      const int t128 = (warp - (3 + EPI_WARPS)) * 32 + lane;
      uint32_t sa = 0, pa = 0, sl = 0, pl = 0;
      // blend one cell (packed fp32x2 math: t = a + w (b - a), so that w = 0 / 1 copy a / b): chunk k of cell (cm, cn)
      auto blend_cell = [&](uint32_t lbase, uint32_t abase, uint32_t k, int cm, int cn, float wy0, float wy1, float wx0, float wx1) {
        // the low-resolution window is NOT swizzled (its tensor map says so): the eight lanes of a cell read one pixel's
        // 128 contiguous bytes, which is conflict-free as it is, and the four corners are constant offsets from one address
        const uint32_t pa = lbase + (cm * LP + cn) * 128 + (k << 4);
        uint32_t a[4], bq[4], c[4], d[4];
        ld_shared_u4(pa, a[0], a[1], a[2], a[3]);
        ld_shared_u4(pa + 128, bq[0], bq[1], bq[2], bq[3]);
        ld_shared_u4(pa + LP * 128, c[0], c[1], c[2], c[3]);
        ld_shared_u4(pa + LP * 128 + 128, d[0], d[1], d[2], d[3]);
        uint32_t o00[4], o01[4], o10[4], o11[4];
#pragma unroll
        for (int w = 0; w < 4; ++w) {
          const float al = __uint_as_float(a[w] << 16), ah = __uint_as_float(a[w] & 0xffff0000u);
          const float bl = __uint_as_float(bq[w] << 16), bh = __uint_as_float(bq[w] & 0xffff0000u);
          const float cl = __uint_as_float(c[w] << 16), ch = __uint_as_float(c[w] & 0xffff0000u);
          const float dl = __uint_as_float(d[w] << 16), dh = __uint_as_float(d[w] & 0xffff0000u);
          float el, eh, fl, fh, t0l, t0h, t1l, t1h, u0l, u0h, u1l, u1h, gl, gh, hl, hh, r0, r1;
          add2(el, eh, bl, bh, -al, -ah);                       // b - a   (upper low-resolution row)
          add2(fl, fh, dl, dh, -cl, -ch);                       // d - c   (lower row)
          fma2(t0l, t0h, wx0, wx0, el, eh, al, ah);             // window column 2 cn
          fma2(t1l, t1h, wx1, wx1, el, eh, al, ah);             // window column 2 cn + 1
          fma2(u0l, u0h, wx0, wx0, fl, fh, cl, ch);
          fma2(u1l, u1h, wx1, wx1, fl, fh, cl, ch);
          add2(gl, gh, u0l, u0h, -t0l, -t0h);
          add2(hl, hh, u1l, u1h, -t1l, -t1h);
          fma2(r0, r1, wy0, wy0, gl, gh, t0l, t0h); o00[w] = pack_bf16x2(r0, r1);
          fma2(r0, r1, wy0, wy0, hl, hh, t1l, t1h); o01[w] = pack_bf16x2(r0, r1);
          fma2(r0, r1, wy1, wy1, gl, gh, t0l, t0h); o10[w] = pack_bf16x2(r0, r1);
          fma2(r0, r1, wy1, wy1, hl, hh, t1l, t1h); o11[w] = pack_bf16x2(r0, r1);
        }
        const uint32_t q00 = (2 * cm) * P + 2 * cn, q01 = q00 + 1, q10 = q00 + P, q11 = q10 + 1;
        st_shared_u4(abase + q00 * 128 + ((k ^ (q00 & 7)) << 4), o00[0], o00[1], o00[2], o00[3]);
        st_shared_u4(abase + q01 * 128 + ((k ^ (q01 & 7)) << 4), o01[0], o01[1], o01[2], o01[3]);
        st_shared_u4(abase + q10 * 128 + ((k ^ (q10 & 7)) << 4), o10[0], o10[1], o10[2], o10[3]);
        st_shared_u4(abase + q11 * 128 + ((k ^ (q11 & 7)) << 4), o11[0], o11[1], o11[2], o11[3]);
      };
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        int mt, nt;
        tile_to_mn<CG>(tile, p.n_ntiles, mt, nt);
        const int t = mt % p.tiles_per_img;
        const int ty = t / p.tiles_x, tx = t - ty * p.tiles_x;
        // weight of the SECOND low-resolution row / column for window rows / columns (2 c, 2 c + 1): (1/4, 3/4); on the
        // image edge (first / last cell of a border tile) the pair is a plain copy of (first, second): (0, 1)
        const int edge_r0 = ty == 0 ? 0 : -1, edge_r1 = ty == p.H / 16 - 1 ? 8 : -1;
        const int edge_c0 = tx == 0 ? 0 : -1, edge_c1 = tx == p.tiles_x - 1 ? CW - 1 : -1;
        for (int src = 0; src < p.nsrc; ++src)
          for (int cb = 0; cb < p.cblk[src]; ++cb) {
            const bool tail = cb == p.cblk[src] - 1 && p.ctail[src];   // 32 real channels: chunks 0..3 only
            ptx::mbar_wait_sleep(ptx::smem_u32(&bars.fullL[sl]), pl);         // (polls with a back-off: these warps have slack,
            ptx::mbar_wait_sleep(ptx::smem_u32(&bars.emptyA[sa]), pa ^ 1);    //  the issue slots belong to the epilogue warps)
            const uint32_t lbase = l_ring + sl * p.l_bytes, abase = smem_base + sa * p.a_bytes;
            if (!(p.debug & 64)) {   // (debug bit 64, timing experiments only: windows left stale)
              // thread = (16-byte channel chunk, cell slot): 8 chunks x 16 slots, or 4 chunks x 32 slots for a half block
              const uint32_t k = tail ? (t128 & 3) : (t128 & 7);
              const int slot = tail ? (t128 >> 2) : (t128 >> 3), nslot = tail ? 32 : 16;
              for (int ci = slot; ci < 9 * CW; ci += nslot) {
                const int cm = ci / CW, cn = ci - cm * CW;
                const bool ey = cm == edge_r0 || cm == edge_r1, ex = cn == edge_c0 || cn == edge_c1;
                blend_cell(lbase, abase, k, cm, cn, ey ? 0.f : 0.25f, ey ? 1.f : 0.75f, ex ? 0.f : 0.25f, ex ? 1.f : 0.75f);
              }
            }
            ptx::fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
              ptx::mbar_arrive(ptx::smem_u32(&bars.emptyL[sl]));
              ptx::mbar_arrive_release_rank0(ptx::smem_u32(&bars.fullA[sa]));   // the LEADER's barrier (its MMAs read both windows)
            }
            if (++sl == static_cast<uint32_t>(p.l_stages)) { sl = 0; pl ^= 1; }
            if (++sa == static_cast<uint32_t>(p.a_stages)) { sa = 0; pa ^= 1; }
          }
      }
    }
  } else if (warp >= 2 && warp < 2 + EPI_WARPS) {
    // ============================== epilogue (2 groups x 8 warps) ================
    // What the clock64 profile (TCS_DEBUG=128) showed: the epilogue of a tile is a chain of latencies (TMEM loads of
    // ~1k cycles each while the MMAs run, the GroupNorm exchange between the CTAs of an image, MUFU, proxy fence + TMA
    // stores: ~12k cycles on a K = 864 layer), not of instruction issue, and it does not shrink when the tile is spread
    // over more warps.  So two tiles are kept in flight: group g = 0/1 owns TMEM accumulator set g and therefore every
    // second tile of this CTA, and inside a group warp (q, h) = (TMEM lane quarter, unit) streams its 32 rows x 96
    // columns through registers 32 columns at a time with the next tcgen05.ld already in flight (pass 1: statistics,
    // pass 2: normalise + store).  A group has two tile periods for its epilogue.
    // unit h: MSUB == 2 -> 128-row sub-tile h (all N = 96 channels); MSUB == 1 -> channel half h of the N = 192 tile.
    const int e = warp - 2, grp = e / GRP_WARPS, ew = e % GRP_WARPS, q = warp & 3, h = ew >> 2;
    const int row = q * 32 + lane;
    const int HW = p.H * p.W;
    const int Wp = p.W + 2, Hp = p.H + 2;
    (void)Hp; (void)Wp; (void)HW;
    const uint32_t acc = grp;
    uint32_t acc_phase = 0, slab_buf = 0;
    (void)slab_buf;
    EpiGroupSmem* gsm = &fs->grp[grp];
    (void)gsm;
    const uint32_t slab = slab_base + static_cast<uint32_t>(e) * WARP_SLAB;          // this warp's 2 x 2 KB staging halves
    const bool use_tma_out = !(p.debug & 4);
    const int h16 = p.W == 16 ? p.H : 0;       // 16-pixel rows: a 32-lane block spans two image rows
    (void)h16;
    (void)use_tma_out; (void)slab;
    const int sub = (MSUB == 2) ? h : 0;
    const int col0 = (MSUB == 2) ? 0 : h * UC;   // first channel (inside the N tile) of this warp's columns
    // accumulator row -> pixel.  GEO 0: a sub-tile is 128 consecutive pixels of the image in row-major order;
    // GEO 1: a sub-tile is 16 image rows x 8 pixels (row i -> image row i / 8, pixel i % 8 of the sub-tile's 8)
    auto pixel_of = [&](int mt_, int& img_, int& y_, int& x_) {
      if (GEO == 1) {
        img_ = mt_ / p.tiles_per_img;
        const int t_ = mt_ - img_ * p.tiles_per_img;
        const int ty_ = t_ / p.tiles_x, tx_ = t_ - ty_ * p.tiles_x;
        y_ = ty_ * 16 + (row >> 3);
        x_ = (tx_ * MSUB + sub) * 8 + (row & 7);
      } else {
        const int m_ = (mt_ * MSUB + sub) * 128 + row;
        img_ = m_ / HW;
        const int rem_ = m_ - img_ * HW;
        y_ = rem_ / p.W;
        x_ = rem_ - y_ * p.W;
      }
    };
    uint32_t it = 0;
    const bool prof = TCS_KERNEL_PROFILE && (p.debug & 128) && blockIdx.x == 0 && e == 0;
    long long pw_full = 0, p_ld = 0, p_a = 0, p_b = 0, p_c = 0, pc0 = 0, pc1 = 0, q_post = 0, q_poll = 0, q_npoll = 0, r_math = 0;
    (void)p_ld;
    long long tacc[3] = {0, 0, 0};
    auto release_tmem = [&]() {
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (CG == 2) ptx::mbar_arrive_rank0(ptx::smem_u32(&bars.tmem_empty[acc]));   // the leader's MMA warp waits on it
        else ptx::mbar_arrive(ptx::smem_u32(&bars.tmem_empty[acc]));
      }
    };
    for (int tile = blockIdx.x + grp * gridDim.x; tile < n_tiles; tile += 2 * gridDim.x, acc_phase ^= 1, ++it) {
      int mt, nt;
      tile_to_mn<CG>(tile, p.n_ntiles, mt, nt);
      const uint32_t tbase = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * ACC_STRIDE;
      const uint32_t taddr = tbase + h * UC;
      if (prof) { pc1 = clock64(); if (it) p_c += pc1 - pc0; pc0 = pc1; }
      ptx::mbar_wait(ptx::smem_u32(&bars.tmem_full[acc]), acc_phase);
      ptx::tc_fence_after();
      if (prof) { pc1 = clock64(); pw_full += pc1 - pc0; pc0 = pc1; }
      if (p.debug & 16) { release_tmem(); continue; }   // experiment: no epilogue work at all

      if constexpr (EPI == EPI_EPS) {
        // ---- 96 -> 1 output conv: column 0 of each sub-tile's accumulator is eps; CFG combine in registers
        float e0 = 0.f, e1 = 0.f;
        if (h == 0) {
          if (p.kxn) {
            // columns 0..2 = the kx taps evaluated at THIS pixel's window; eps(x) = c0(x-1) + c1(x) + c2(x+1), circular in
            // x.  A warp holds 32 consecutive pixels of a 64-pixel image row, its partner (q ^ 1) the other half.
            float a0[4], a1[4];
            ptx::tmem_ld4(tbase, a0);
            ptx::tmem_ld4(tbase + N, a1);
            ptx::tmem_ld_wait();
            release_tmem();
            float* xch = reinterpret_cast<float*>(fs) + grp * 32;   // [4 warps][4] exchange slots (EPI_EPS never uses fs otherwise)
            const int qq = q;   // pixel position inside the sub-tile follows the TMEM lane quarter
            if (lane == 31) { xch[qq * 4 + 0] = a0[0]; xch[qq * 4 + 1] = a1[0]; }
            if (lane == 0) { xch[qq * 4 + 2] = a0[2]; xch[qq * 4 + 3] = a1[2]; }
            asm volatile("bar.sync %0, 128;" ::"r"(3 + grp) : "memory");
            float l0 = __shfl_up_sync(0xffffffffu, a0[0], 1), l1 = __shfl_up_sync(0xffffffffu, a1[0], 1);
            float r0 = __shfl_down_sync(0xffffffffu, a0[2], 1), r1 = __shfl_down_sync(0xffffffffu, a1[2], 1);
            const int pq = qq ^ 1;
            if (lane == 0) { l0 = xch[pq * 4 + 0]; l1 = xch[pq * 4 + 1]; }
            if (lane == 31) { r0 = xch[pq * 4 + 2]; r1 = xch[pq * 4 + 3]; }
            e0 = (l0 + a0[1]) + r0;
            e1 = (l1 + a1[1]) + r1;
            asm volatile("bar.sync %0, 128;" ::"r"(3 + grp) : "memory");   // slots are free for the next tile
          } else {
            ptx::tmem_ld1(tbase, &e0);
            ptx::tmem_ld1(tbase + N, &e1);
            ptx::tmem_ld_wait();
            release_tmem();
          }
        } else {
          release_tmem();
        }
        if (h == 0) {
          e0 += bias_s[0];
          e1 += bias_s[0];
          float* eo = static_cast<float*>(p.epi.out);
          if (p.pair) {          // sub-tile 0 = conditional image 2i, sub-tile 1 = unconditional image 2i+1
            eo[static_cast<size_t>(mt) * 128 + row] = e1 + p.guidance * (e0 - e1);
          } else {
            eo[static_cast<size_t>(mt) * 256 + row] = e0;
            eo[static_cast<size_t>(mt) * 256 + 128 + row] = e1;
          }
        }
      } else if constexpr (EPI == EPI_GN_FUSED) {
        // ---- conv + bias + GroupNorm + SiLU without leaving TMEM ------------------------------------------------
        // The G = tiles_per_img CTAs with blockIdx % G == 0..G-1 hold one image between them and run it in lock
        // step: per-group sums of this CTA's pixels -> global, wait for the other G-1 CTAs, then normalise + SiLU
        // straight from TMEM.
        constexpr int CPGN = N / 8;            // channels per group: 12 or 24
        constexpr int NGL = UC / CPGN;         // groups inside this warp's columns: 8 or 4
        const int G = p.tiles_per_img;
        const int img = mt / G;
        float rv[2 * NGL];                     // (sum, sum of squares) per local group
        // Pass 1 reads the accumulator ONCE (32 columns at a time, next tcgen05.ld in flight): statistics in fp32, and the
        // biased values (bias_s holds bias - K_g, see its load) are kept as fp16 (3 more mantissa bits than the bf16 output,
        // satfinite): column blocks 0 and 1 in
        // this warp's two output staging blocks (same [32 px][64 B] swizzled rows as the bf16 output that replaces them in
        // place in pass 2; a lane only ever touches its own row), block 2 in 16 registers.  The TMEM set therefore goes
        // back to the MMA warps BEFORE the cross-CTA exchange (the accumulator hold time was the bound of the K = 864
        // layers: ~10k cycles against ~6k of MMA work per tile).
        uint32_t stash2[BLK / 2];
        const uint32_t srow = slab + lane * 64;        // this lane's row inside a staging block
        const int ssw = (lane >> 1) & 3;
        const uint32_t sb0 = slab_buf;                 // staging block that pass 2 fills first
        // TCS_STASH_TMEM (default): column blocks 0 and 1 of the stash live in the 64 TMEM columns an accumulator set
        // leaves free (192 of 256), 32 per warp unit, instead of the staging blocks: tcgen05.st / ld do not touch shared
        // memory, whose bandwidth the MMA operand reads of an N = 96 layer already use to ~90 %
        const bool stash_tmem = !(p.debug & 32);
        const uint32_t tstash = tbase + N * MSUB + h * 32;
        if (use_tma_out && !stash_tmem) {              // the previous tile's TMA stores have left the staging blocks
          const long long cl0 = prof ? clock64() : 0;
          if (lane == 0) ptx::bulk_wait_read<0>();
          __syncwarp();
          if (prof) p_ld += clock64() - cl0;
        }
        {
          float gs[NGL], gq[NGL];
#pragma unroll
          for (int g = 0; g < NGL; ++g) gs[g] = gq[g] = 0.f;
          float vbuf[2][32];
          ptx::tmem_ld32(taddr, vbuf[0]);
#pragma unroll
          for (int k = 0; k < 3; ++k) {
            ptx::tmem_ld_wait();
            if (k < 2) ptx::tmem_ld32(taddr + (k + 1) * 32, vbuf[(k + 1) & 1]);
            else release_tmem();
            const float* v = vbuf[k & 1];
            const uint32_t sblk = srow + ((sb0 ^ (k & 1)) * 2048);
#pragma unroll
            for (int i = 0; i < 32; i += 8) {
              uint32_t hw[4];
#pragma unroll
              for (int u = 0; u < 8; u += 4) {
                const float4 b4 = *reinterpret_cast<const float4*>(bias_s + col0 + k * 32 + i + u);
                float t0, t1, t2, t3;
                add2(t0, t1, v[i + u], v[i + u + 1], b4.x, b4.y);
                add2(t2, t3, v[i + u + 2], v[i + u + 3], b4.z, b4.w);
                const int g0 = (k * 32 + i + u) / CPGN, g1 = (k * 32 + i + u + 2) / CPGN;   // pairs never straddle a group
                gs[g0] += t0; gq[g0] = fmaf(t0, t0, gq[g0]);
                gs[g0] += t1; gq[g0] = fmaf(t1, t1, gq[g0]);
                gs[g1] += t2; gq[g1] = fmaf(t2, t2, gq[g1]);
                gs[g1] += t3; gq[g1] = fmaf(t3, t3, gq[g1]);
                hw[u / 2] = pack_f16x2_sat(t0, t1);
                hw[u / 2 + 1] = pack_f16x2_sat(t2, t3);
              }
              if (k < 2 && !stash_tmem) {
                st_shared_u4(sblk + (((i / 8) ^ ssw) << 4), hw[0], hw[1], hw[2], hw[3]);
              } else {
#pragma unroll
                for (int u = 0; u < 4; ++u) stash2[i / 2 + u] = hw[u];
              }
            }
            if (k < 2 && stash_tmem) ptx::tmem_st16(tstash + k * 16, stash2);
          }
          if (stash_tmem) ptx::tmem_st_wait();
          // fp16 stash range guard, for free: a row whose sum of squares over a group stays below 65504^2 cannot hold a
          // value that saturated in cvt.rn.satfinite.  Otherwise flag the launch: the host re-runs the evaluation on the
          // unfused path (conv -> fp32 -> GroupNorm kernel) instead of returning a clipped activation.
          bool ovf = false;
#pragma unroll
          for (int g = 0; g < NGL; ++g) { rv[2 * g] = gs[g]; rv[2 * g + 1] = gq[g]; ovf |= !(gq[g] < 4.2907e9f); }
          if (__any_sync(0xffffffffu, ovf) && lane == 0 && p.epi.overflow) atomicOr(p.epi.overflow, 1);
        }
        // lane reduction: a reduce-scatter over the top lane bits (2*NGL values -> 1 per lane), butterflies for the rest
        constexpr int NV = 2 * NGL;            // 8 or 16
        constexpr int SC_STEPS = NV == 16 ? 4 : 3;
        int idx = 0;
#pragma unroll
        for (int st = 0; st < SC_STEPS; ++st) {
          const int half = NV >> (st + 1), off = 16 >> st;
          const bool hi = (lane & off) != 0;
#pragma unroll
          for (int i = 0; i < half; ++i) {
            const float send = hi ? rv[i] : rv[i + half];
            const float keep = hi ? rv[i + half] : rv[i];
            rv[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
          }
          idx |= hi ? half : 0;
        }
#pragma unroll
        for (int off = 16 >> SC_STEPS; off >= 1; off >>= 1) rv[0] += __shfl_xor_sync(0xffffffffu, rv[0], off);
        if (lane < 16) gsm->red[ew][lane] = 0.f;   // the slots of the groups this warp does not cover
        __syncwarp();
        if ((lane & ((32 >> SC_STEPS) - 1)) == 0) gsm->red[ew][2 * (col0 / CPGN) + idx] = rv[0];
        epi_bar_sync(grp);
        if (prof) { pc1 = clock64(); p_a += pc1 - pc0; pc0 = pc1; }
        if (ew == 0) {
          // Exchange between the G CTAs of the image, one L2 round trip each way: every (value, flag) pair is ONE 64-bit
          // word (the flag travels with the data, as in NCCL's LL protocol), so there is no separate counter, no fence and
          // no second read.  The buffer is zeroed before the launch; flag 1 = valid.
          unsigned long long* ll = reinterpret_cast<unsigned long long*>(p.epi.partials);
          if (lane < 16) {
            float tot = 0.f;
#pragma unroll
            for (int w = 0; w < GRP_WARPS; ++w) tot += gsm->red[w][lane];
            st_relaxed_gpu_u64(ll + static_cast<size_t>(mt) * 16 + lane, (1ULL << 32) | __float_as_uint(tot));
          }
          if (prof) { pc1 = clock64(); q_post += pc1 - pc0; }
          // 16 values x G CTAs: lane l sums value (l & 15) over the CTAs of parity (l >> 4), fixed order
          const unsigned long long* ip = ll + static_cast<size_t>(img) * G * 16 + (lane & 15);
          float part = 0.f;
          {
            const long long t0 = clock64();
            int polls = 0;
            unsigned long long w[8];        // G <= 16: at most 8 words per lane, all loads in flight together
            bool ready;
            do {
              ready = true;
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                const int k = (lane >> 4) + 2 * i;
                w[i] = k < G ? ld_relaxed_gpu_u64(ip + k * 16) : (1ULL << 32);
              }
#pragma unroll
              for (int i = 0; i < 8; ++i) ready = ready && ((w[i] >> 32) == 1ULL);
              if (p.debug & 1) ready = true;
              if (!ready) {
                ++polls;
                if (clock64() - t0 > p.exch_timeout) __trap();   // -> launch failure, reported as TCS_ERR_CUDA
              }
            } while (!ready);
#pragma unroll
            for (int i = 0; i < 8; ++i) part += __uint_as_float(static_cast<uint32_t>(w[i]));   // zeros for k >= G
            if (prof) { q_poll += clock64() - pc1; q_npoll += polls; }
          }
          part += __shfl_xor_sync(0xffffffffu, part, 16);
          const float qsum = __shfl_down_sync(0xffffffffu, part, 1);   // lane 2g: sum, lane 2g+1: sum of squares
          if (lane < 16 && (lane & 1) == 0) {
            // no double-precision DIVIDE here: on this part it is a long software routine on the critical path of the
            // whole image group (measured: ~4k cycles per tile); 1/count comes from the host
            const double mean = static_cast<double>(part) * p.gn_inv_cnt;
            double var = fma(-mean, mean, static_cast<double>(qsum) * p.gn_inv_cnt);
            var = var < 0.0 ? 0.0 : var;
            gsm->mean[lane >> 1] = static_cast<float>(mean);
            gsm->rstd[lane >> 1] = rsqrtf(static_cast<float>(var) + GN_EPS);
          }
          __syncwarp();
          for (int c = lane; c < N; c += 32) {      // per-channel affine table, by the same warp (saves a group barrier)
            const int g = c / CPGN;
            const float sc = gsm->rstd[g] * fs->gamma[c];
            gsm->scale[c] = 0.5f * sc;                                                  // h = y / 2 = v * scale + shift
            gsm->shift[c] = 0.5f * (fs->beta[c] - gsm->mean[g] * sc);                   // mean and stash both exclude K_g
          }
        }
        epi_bar_sync(grp);
        if (prof) { pc1 = clock64(); p_b += pc1 - pc0; pc0 = pc1; }
        __nv_bfloat16* obase = static_cast<__nv_bfloat16*>(p.epi.out);
        int img_px, y, x;
        pixel_of(mt, img_px, y, x);
        (void)img_px;
        const int wy = (y == 0) ? p.H : ((y == p.H - 1) ? -p.H : 0);
        const int wx = (x == 0) ? p.W : ((x == p.W - 1) ? -p.W : 0);
        const size_t pix = (static_cast<size_t>(img) * Hp + (y + 1)) * Wp + (x + 1);
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          const int cc = col0 + k * 32;
          uint32_t hv[16];
          if (k < 2 && stash_tmem) {
            ptx::tmem_ld16(tstash + k * 16, reinterpret_cast<float*>(hv));
            ptx::tmem_ld_wait();
          } else if (k < 2) {
            const uint32_t sblk = srow + ((sb0 ^ k) * 2048);   // = the block store_padded_block fills next (in place)
#pragma unroll
            for (int j = 0; j < 4; ++j) ld_shared_u4(sblk + ((j ^ ssw) << 4), hv[4 * j], hv[4 * j + 1], hv[4 * j + 2], hv[4 * j + 3]);
          } else {
#pragma unroll
            for (int j = 0; j < 16; ++j) hv[j] = stash2[j];
          }
          uint32_t pk[16];
#pragma unroll
          for (int i = 0; i < 32; i += 4) {
            const float4 s4 = *reinterpret_cast<const float4*>(gsm->scale + cc + i);
            const float4 h4 = *reinterpret_cast<const float4*>(gsm->shift + cc + i);
            const float2 va = unpack_f16x2(hv[i / 2]), vb = unpack_f16x2(hv[i / 2 + 1]);
            float h0, h1, h2, h3, y0, y1, y2, y3;
            fma2(h0, h1, va.x, va.y, s4.x, s4.y, h4.x, h4.y);              // h = y/2
            fma2(h2, h3, vb.x, vb.y, s4.z, s4.w, h4.z, h4.w);
            fma2(y0, y1, h0, h1, tanh_fast(h0), tanh_fast(h1), h0, h1);    // SiLU(y) = h + h tanh(h)
            fma2(y2, y3, h2, h3, tanh_fast(h2), tanh_fast(h3), h2, h3);
            pk[i / 2] = pack_bf16x2(y0, y1);
            pk[i / 2 + 1] = pack_bf16x2(y2, y3);
          }
          if (!(p.debug & 2))
            store_padded_block<GEO>(&mapO, use_tma_out, slab, slab_buf, lane, obase, pix, wy, wx, Wp, p.epi.ldo, cc, img, y, x, pk,
                                    prof ? tacc : nullptr, GEO == 1 ? 0 : h16, &mapO1, p.H);
          else if (pk[0] == 0x12345678u && pk[7] == 0x9abcdef0u) obase[0] = __float2bfloat16(0.f);
        }
        if (prof) r_math += clock64() - pc1;
      } else if constexpr (N >= 96) {
        const int n_off = nt * N + col0;                     // first output channel of this warp's columns
        int b, y, x;
        pixel_of(mt, b, y, x);
        const int m = (b * p.H + y) * p.W + x;               // global pixel index (b, y, x)
        float vbuf[2][32];
        ptx::tmem_ld32(taddr, vbuf[0]);
        if constexpr (EPI == EPI_RAW_STATS) {
          // fp32 output (one row per lane, plain stores) plus per-(warp, group) partial sums for a separate GroupNorm
          // pass: the unfused A/B path (TCS_FUSE_GN=0) and the per-layer tests; not on the production path
          constexpr int CPGN = N / 8;
          constexpr int NG = UC / CPGN;
          float gs[NG], gq[NG];
#pragma unroll
          for (int g = 0; g < NG; ++g) gs[g] = gq[g] = 0.f;
          float* orow = static_cast<float*>(p.epi.out) + static_cast<size_t>(m) * p.epi.ldo + n_off;
#pragma unroll
          for (int k = 0; k < 3; ++k) {
            ptx::tmem_ld_wait();
            if (k < 2) ptx::tmem_ld32(taddr + (k + 1) * 32, vbuf[(k + 1) & 1]);
            else release_tmem();
            float* v = vbuf[k & 1];
#pragma unroll
            for (int i = 0; i < 32; i += 4) {
              const float4 b4 = *reinterpret_cast<const float4*>(bias_s + n_off + k * 32 + i);
              v[i] += b4.x; v[i + 1] += b4.y; v[i + 2] += b4.z; v[i + 3] += b4.w;
              *reinterpret_cast<float4*>(orow + k * 32 + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
            }
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              gs[(k * 32 + i) / CPGN] += v[i];
              gq[(k * 32 + i) / CPGN] += v[i] * v[i];
            }
          }
#pragma unroll
          for (int g = 0; g < NG; ++g) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
              gs[g] += __shfl_xor_sync(0xffffffffu, gs[g], o);
              gq[g] += __shfl_xor_sync(0xffffffffu, gq[g], o);
            }
          }
          if (lane == 0) {
            // slot layout [image][tile-in-image*MSUB + sub][quarter]; the column units of a row block write disjoint
            // groups of the same slot
            const int slot = ((mt * MSUB + sub) % (p.tiles_per_img * MSUB)) * 4 + q;
            float* dst = p.epi.partials + (static_cast<size_t>(b) * p.epi.slots + slot) * 16 + 2 * (col0 / CPGN);
#pragma unroll
            for (int g = 0; g < NG; ++g) { dst[2 * g] = gs[g]; dst[2 * g + 1] = gq[g]; }
          }
        } else if constexpr (EPI == EPI_PADDED) {
          const int wy = (y == 0) ? p.H : ((y == p.H - 1) ? -p.H : 0);
          const int wx = (x == 0) ? p.W : ((x == p.W - 1) ? -p.W : 0);
          __nv_bfloat16* obase = static_cast<__nv_bfloat16*>(p.epi.out);
          const size_t pix = (static_cast<size_t>(b) * Hp + (y + 1)) * Wp + (x + 1);
          const __nv_bfloat16* rrow =
              p.epi.residual ? static_cast<const __nv_bfloat16*>(p.epi.residual) + pix * p.ntot + n_off : nullptr;
#pragma unroll
          for (int k = 0; k < 3; ++k) {
            const int c0 = k * 32;
            ptx::tmem_ld_wait();
            if (k < 2) ptx::tmem_ld32(taddr + (k + 1) * 32, vbuf[(k + 1) & 1]);
            else release_tmem();
            float* v = vbuf[k & 1];
            if (rrow) {
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const uint4 rr = *reinterpret_cast<const uint4*>(rrow + c0 + i * 8);
                const uint32_t w4[4] = {rr.x, rr.y, rr.z, rr.w};
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {
                  const float2 rf = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w4[kk]));
                  v[i * 8 + 2 * kk] += rf.x;
                  v[i * 8 + 2 * kk + 1] += rf.y;
                }
              }
            }
            uint32_t pk[16];
#pragma unroll
            for (int i = 0; i < 32; i += 4) {
              const float4 b4 = *reinterpret_cast<const float4*>(bias_s + n_off + c0 + i);
              pk[i / 2] = pack_bf16x2(v[i] + b4.x, v[i + 1] + b4.y);
              pk[i / 2 + 1] = pack_bf16x2(v[i + 2] + b4.z, v[i + 3] + b4.w);
            }
            store_padded_block<GEO, SB>(&mapO, use_tma_out, slab, slab_buf, lane, obase, pix, wy, wx, Wp, p.epi.ldo, n_off + c0, b, y, x, pk,
                                        nullptr, GEO == 1 ? 0 : h16, &mapO1, p.H);
          }
        } else {  // EPI_PLAIN: unpadded bf16 [pixel][ldo] rows; 32 px x 32 ch blocks staged in the warp's slabs and
                  // TMA-stored (a lane-per-row 16-byte store touches 32 different lines per instruction)
          __nv_bfloat16* orow = static_cast<__nv_bfloat16*>(p.epi.out) + static_cast<size_t>(m) * p.epi.ldo + n_off;
          const bool tma_plain = !(p.debug & 4);
#pragma unroll
          for (int k = 0; k < 3; ++k) {
            ptx::tmem_ld_wait();
            if (k < 2) ptx::tmem_ld32(taddr + (k + 1) * 32, vbuf[(k + 1) & 1]);
            else release_tmem();
            const float* v = vbuf[k & 1];
            uint32_t pk[16];
#pragma unroll
            for (int i = 0; i < 32; i += 4) {
              const float4 b4 = *reinterpret_cast<const float4*>(bias_s + n_off + k * 32 + i);
              pk[i / 2] = pack_bf16x2(v[i] + b4.x, v[i + 1] + b4.y);
              pk[i / 2 + 1] = pack_bf16x2(v[i + 2] + b4.z, v[i + 3] + b4.w);
            }
            if (tma_plain) {
              if (lane == 0) ptx::bulk_wait_read<SLAB_BUFS - 1>();
              __syncwarp();
              const uint32_t base = slab + (SLAB_BUFS == 2 ? slab_buf * 2048 : 0);
              const uint32_t dst = base + lane * 64;
              const int sw = (lane >> 1) & 3;
#pragma unroll
              for (int j = 0; j < 4; ++j) st_shared_u4(dst + ((j ^ sw) << 4), pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
              ptx::fence_proxy_async();
              __syncwarp();
              if (lane == 0) {
                ptx::tma_store_2d(&mapO, base, n_off + k * 32, m - lane);   // rows m - lane .. m - lane + 31 of the [M, ldo] tensor
                ptx::bulk_commit();
              }
              slab_buf ^= 1;
            } else {
#pragma unroll
              for (int i = 0; i < 4; ++i)
                *reinterpret_cast<uint4*>(orow + k * 32 + i * 8) = make_uint4(pk[4 * i], pk[4 * i + 1], pk[4 * i + 2], pk[4 * i + 3]);
            }
          }
        }
      }
    }
    if (prof && lane == 0 && it > 1)
      printf("[epi N=%d EPI=%d] per tile: wait tmem_full %lld  staging-block wait %lld  pass1+barA %lld  exchange+table+barB %lld (post %lld, poll %lld, polls %lld)  pass2+stores+loop %lld (pass2 %lld: wait_read %lld, sts+fence %lld, tma issue %lld)\n",
             N, EPI, pw_full / it, p_ld / it, p_a / it, p_b / it, q_post / it, q_poll / it, q_npoll / it, p_c / (it - 1), r_math / it, tacc[0] / it, tacc[1] / it, tacc[2] / it);
    if (lane == 0) ptx::bulk_wait_all();   // staged TMA stores have left shared memory
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (CG == 2) ptx::cluster_sync_all();   // the leader's MMAs read the peer's shared memory / write its TMEM
  ptx::tc_fence_after();
  if (warp == 1) {
    if (CG == 2) ptx::tmem_dealloc_512_2sm(tmem_base);
    else ptx::tmem_dealloc_512(tmem_base);
  }
}

// ---------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------
static void stage_shape(const ConvGeom& g, int* T, int* KYG, int* KW) {
  *KW = g.kx_in_n ? 1 : g.ksize;
  if (g.ksize == 4) { *T = 2; *KYG = 2; }
  else if (g.ksize == 3) { *T = 3; *KYG = 1; }
  else { *T = 1; *KYG = 1; }
}

int conv_tc_kstages(const ConvGeom& g) {
  int T, KYG, KW;
  stage_shape(g, &T, &KYG, &KW);
  int cb = 0;
  for (int s = 0; s < g.nsrc; ++s) cb += (g.csrc[s] + KB - 1) / KB;
  return cb * KYG * KW * (g.split3 ? 3 : 1);
}

size_t conv_tc_packed_elems(const ConvGeom& g) {
  int T, KYG, KW;
  stage_shape(g, &T, &KYG, &KW);
  return static_cast<size_t>(conv_tc_kstages(g)) * T * g.ntot * KB;
}

// N tile and CTA-pair choice of a layer (shared by the weight packer and the plan)
void conv_tc_tile_shape(const ConvGeom& g, int epi, int* N, int* cg) {
  *N = (epi == EPI_EPS) ? 16 : ((g.ntot % 192 == 0) ? 192 : 96);
  const char* e = getenv("TCS_CG");   // 1 = single-CTA MMA everywhere (A/B switch)
  *cg = (*N >= 96 && !(e && atoi(e) == 1)) ? 2 : 1;
  // (with 64-channel K blocks a single CTA cannot hold two stages of a whole weight tile of a 3x3 / 4x4 layer: under
  // the switch only the 1x1 layers and the output conv run single-CTA MMAs)
  if (*N >= 96 && g.ksize >= 3) *cg = 2;
  // the 96 -> 1 output conv is bound by MMA ISSUE (36 tiny N = 16 MMAs per tile at ~100 cycles each): as a CTA pair one
  // thread's MMA covers both CTAs' tiles, which halves the issue work per tile
  const char* e2 = getenv("TCS_EPS_CG");
  if (epi == EPI_EPS && !(e && atoi(e) == 1) && !(e2 && atoi(e2) == 1)) *cg = 2;
}

// Packed layout: [K stage][N tile][CTA of the pair][tap][N/cg rows][64 channels], every 128-byte row with its 16-byte
// chunks permuted as SWIZZLE_128B would place them (chunk ^ (row & 7)), i.e. the shared-memory image itself, so that TMA
// can move a stage's weights as one box of 512-byte rows without swizzling.  Channels past the end of a source (the
// upper half of the block that ends a 96-channel source) are zero and never read by the MMAs.
void conv_tc_pack_weights(const ConvGeom& g, int epi, const float* w, __nv_bfloat16* out) {
  int T, KYG, KW, N, cg;
  stage_shape(g, &T, &KYG, &KW);
  conv_tc_tile_shape(g, epi, &N, &cg);
  const int NB = N / cg, n_ntiles = g.ntot / N;
  const int k = g.ksize;
  int cin_tot = 0;
  for (int s = 0; s < g.nsrc; ++s) cin_tot += g.csrc[s];
  size_t ks = 0;
  int coff = 0;
  const int nseg = g.split3 ? 3 : 1;          // K segments per logical source: [w_hi, w_lo, w_hi] against [a_hi, a_hi, a_lo]
  for (int s = 0; s < g.nsrc; ++s) {
    for (int seg = 0; seg < nseg; ++seg)
      for (int cb = 0; cb < (g.csrc[s] + KB - 1) / KB; ++cb)
        for (int kyg = 0; kyg < KYG; ++kyg)
          for (int kx = 0; kx < KW; ++kx, ++ks)
            for (int j = 0; j < T; ++j) {
              const int ky = (g.ksize == 4) ? kyg + 2 * j : j;
              for (int n = 0; n < g.ntot; ++n)
                for (int c = 0; c < KB; ++c) {
                  const int ci = coff + cb * KB + c;
                  float v;
                  if (cb * KB + c >= g.csrc[s]) v = 0.f;
                  else if (g.kx_in_n) v = n < k ? w[((static_cast<size_t>(0) * cin_tot + ci) * k + ky) * k + n] : 0.f;   // column n = tap kx
                  else v = w[((static_cast<size_t>(n) * cin_tot + ci) * k + ky) * k + kx];
                  __nv_bfloat16 hi = __float2bfloat16(v);
                  if (seg == 1) hi = __float2bfloat16(v - __bfloat162float(hi));   // w_lo
                  const int nt = n / N, nn = n % N, half = nn / NB, r = nn % NB;
                  const int pc = (c / 8) ^ (r & 7);
                  out[((((ks * n_ntiles + nt) * cg + half) * T + j) * NB + r) * KB + pc * 8 + (c % 8)] = hi;
                }
            }
    coff += g.csrc[s];
  }
}

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_encodeTiled>(p);
  }
  return fn;
}

// EPI_EPS with CFG: re-shape a plan so that each CTA tile holds the same Rt rows of images 2i and 2i+1
int conv_tc_make_pair(ConvTcPlan* pl, const void* src, int B) {
  ConvTcParams& p = pl->p;
  if (pl->epi != EPI_EPS || pl->msub != 2 || B % 2) return fail(TCS_ERR_BAD_ARGUMENT, "conv_tc_make_pair: needs the eps plan and an even batch");
  PFN_encodeTiled encode = get_encode();
  p.pair = 1;
  p.WR = p.Rt + p.T - 1;
  p.tiles_per_img = p.H / p.Rt;                       // tiles per image PAIR
  p.n_mtiles = (B / 2) * p.tiles_per_img;
  p.a_bytes = 2u * static_cast<uint32_t>(p.WR) * p.W * ROWB;
  p.stage_bytes = (p.a_bytes + p.T * (pl->N / pl->cg) * ROWB + 1023u) & ~1023u;
  const size_t budget = 227 * 1024 - 2048 - 1024 - EPI_SLAB_BYTES - EPI_BIAS_BYTES - EPI_FUSED_BYTES;
  p.nstage = static_cast<int>(budget / p.stage_bytes);
  if (p.nstage > MAX_STAGES) p.nstage = MAX_STAGES;
  pl->smem = static_cast<size_t>(p.nstage) * p.stage_bytes + 1024 + EPI_SLAB_BYTES + EPI_BIAS_BYTES + EPI_FUSED_BYTES;
  const cuuint64_t C = static_cast<cuuint64_t>(pl->cin[0]);
  const int Hin = p.H + 2, Win = p.W + 2;
  cuuint64_t dims[4] = {C, static_cast<cuuint64_t>(Win), static_cast<cuuint64_t>(Hin), static_cast<cuuint64_t>(B)};
  cuuint64_t strides[3] = {C * 2, C * 2 * Win, C * 2 * Win * Hin};
  cuuint32_t box[4] = {KB, static_cast<cuuint32_t>(p.W), static_cast<cuuint32_t>(p.WR), 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = encode(&pl->mapA[0], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(src), dims, strides, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(TCS_ERR_CUDA, "cuTensorMapEncodeTiled(A pair) failed: " + std::to_string(r));
  for (int i = 1; i < 4; ++i) pl->mapA[i] = pl->mapA[0];
  return TCS_OK;
}

int conv_tc_grid(const ConvTcPlan& pl, int B, int sm_count) {
  const int tiles = (pl.p.pair ? B / 2 : B) * pl.p.tiles_per_img * pl.p.n_ntiles;
  int grid = tiles < sm_count ? tiles : sm_count;
  if (pl.max_ctas > 0 && grid > pl.max_ctas) grid = pl.max_ctas;   // what the device can hold at once (occupancy query)
  // Fused GroupNorm: the tiles of an image exchange partial sums through L2 words indexed by TILE, not by CTA, so any
  // co-resident grid is correct and deadlock-free (a tile only ever waits for tiles of its own image, i.e. for tile indices
  // at most one grid-stride ahead, whose CTAs never wait for anything later).  Whole image groups (grid a multiple of the
  // tiles per image) keep every image inside one wave; the full grid lets one image in ~9 straddle two waves (its first
  // tiles' epilogue group waits one tile period, which the other group and the double-buffered accumulators absorb) but
  // uses all SMs: 148 instead of 144 on the 64x64 and 32x32 layers.  TCS_GN_GROUP_GRID=1 restores the rounded grid.
  static const bool group_grid = getenv("TCS_GN_GROUP_GRID") && atoi(getenv("TCS_GN_GROUP_GRID")) == 1;
  if (pl.epi == EPI_GN_FUSED && (group_grid || grid < pl.p.tiles_per_img * 2))
    grid = grid / pl.p.tiles_per_img * pl.p.tiles_per_img;
  if (pl.cg == 2) grid &= ~1;                                                         // whole CTA pairs
  return grid;
}

// Can one launch carry BOTH the cooperative and the cluster attribute?  Probed once with an empty kernel, outside any
// stream capture (a failed launch would invalidate a capture).
__global__ void coop_cluster_probe_kernel() {}
static bool coop_cluster_supported() {
  static int state = -1;
  if (state < 0) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(2); cfg.blockDim = dim3(32); cfg.dynamicSmemBytes = 0; cfg.stream = nullptr;
    cudaLaunchAttribute at[2];
    at[0].id = cudaLaunchAttributeCooperative; at[0].val.cooperative = 1;
    at[1].id = cudaLaunchAttributeClusterDimension;
    at[1].val.clusterDim.x = 2; at[1].val.clusterDim.y = 1; at[1].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 2;
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(nullptr, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone) { cudaGetLastError(); return false; }
    const cudaError_t e = cudaLaunchKernelEx(&cfg, coop_cluster_probe_kernel);
    cudaGetLastError();
    state = (e == cudaSuccess && cudaDeviceSynchronize() == cudaSuccess) ? 1 : 0;
    if (getenv("TCS_NO_COOP_CLUSTER")) state = 0;
  }
  return state == 1;
}

// tap-shift geometry (GEO = 1) for every 3x3 stride-1 layer; TCS_GEO=0 keeps the per-kx row windows (A/B switch)
static int conv_tc_geo(const ConvGeom& g, int epi) {
  const char* e = getenv("TCS_GEO");
  if (e && atoi(e) == 0) return 0;
  return (g.ksize == 3 && g.stride == 1 && !g.kx_in_n && epi != EPI_EPS && epi != EPI_PLAIN && g.H % 16 == 0) ? 1 : 0;
}

template <int N, int EPI, int MSUB, int CG, int GEO, int UPS = 0>
static int set_smem_attr() {
  static bool attr_done = false;
  if (!attr_done) {
    TCS_CUDA(cudaFuncSetAttribute(conv_tc_kernel<N, EPI, MSUB, CG, GEO, UPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(TC_SMEM_MAX)));
    attr_done = true;
  }
  return TCS_OK;
}

// CTAs of this kernel instance the device can hold at the same time (1 CTA per SM by shared memory; with CTA pairs,
// whole clusters only: on a partitioned or partly occupied device fewer pairs fit than SMs / 2)
template <int N, int EPI, int MSUB, int CG, int GEO, int UPS = 0>
static int max_ctas_t(const ConvTcPlan& pl, int* out) {
  TCS_CHECK((set_smem_attr<N, EPI, MSUB, CG, GEO, UPS>()));
  auto kern = conv_tc_kernel<N, EPI, MSUB, CG, GEO, UPS>;
  if (CG == 2) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(2); cfg.blockDim = dim3(TC_THREADS + UPS_EXTRA_THREADS * UPS); cfg.dynamicSmemBytes = pl.smem; cfg.stream = nullptr;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    int nclusters = 0;
    TCS_CUDA(cudaOccupancyMaxActiveClusters(&nclusters, kern, &cfg));
    *out = 2 * nclusters;
  } else {
    int per_sm = 0, dev = 0, sms = 0;
    TCS_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, TC_THREADS, pl.smem));
    TCS_CUDA(cudaGetDevice(&dev));
    TCS_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    *out = per_sm * sms;
  }
  return TCS_OK;
}

template <int N, int EPI, int MSUB, int CG, int GEO, int UPS = 0>
static int launch_t(const ConvTcPlan& pl, cudaStream_t st) {
  auto kern = conv_tc_kernel<N, EPI, MSUB, CG, GEO, UPS>;
  TCS_CHECK((set_smem_attr<N, EPI, MSUB, CG, GEO, UPS>()));
  if (EPI == EPI_GN_FUSED)   // the CTAs of an image group exchange (value, flag) words: flag 0 = not written yet
    TCS_CUDA(cudaMemsetAsync(pl.p.epi.partials, 0, sizeof(unsigned long long) * 16 * pl.p.n_mtiles, st));
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(pl.grid); cfg.blockDim = dim3(TC_THREADS + UPS_EXTRA_THREADS * UPS); cfg.dynamicSmemBytes = pl.smem; cfg.stream = st;
  cudaLaunchAttribute at[2];
  int na = 0;
  // the CTAs of an image group poll each other's partial sums: the whole grid must be co-resident.  The cooperative
  // attribute makes the runtime guarantee it (gang scheduling, also against kernels of other streams); where it cannot
  // be combined with clusters the grid is still <= cudaOccupancyMaxActiveClusters (conv_tc_grid).
  if (EPI == EPI_GN_FUSED && (CG == 1 || pl.coop_cluster)) {
    at[na].id = cudaLaunchAttributeCooperative;
    at[na].val.cooperative = 1;
    ++na;
  }
  if (CG == 2) {
    at[na].id = cudaLaunchAttributeClusterDimension;
    at[na].val.clusterDim.x = 2; at[na].val.clusterDim.y = 1; at[na].val.clusterDim.z = 1;
    ++na;
  }
  cfg.attrs = at; cfg.numAttrs = na;
  TCS_CUDA(cudaLaunchKernelEx(&cfg, kern, pl.mapA[0], pl.mapA[1], pl.mapA[2], pl.mapA[3], pl.mapW, pl.mapO, pl.mapO1, pl.p));
  TCS_CUDA(cudaGetLastError());
  return TCS_OK;
}

static int conv_tc_max_ctas(const ConvTcPlan& pl, int* out) {
#define TCS_TC_CASE(NN, EE, MM)                                                        \
  if (pl.geo == 0 && pl.N == NN && pl.epi == EE && pl.msub == MM) {                     \
    if (pl.cg == 2) { if constexpr (NN >= 96 || EE == EPI_EPS) return max_ctas_t<NN, EE, MM, 2, 0>(pl, out); } \
    else return max_ctas_t<NN, EE, MM, 1, 0>(pl, out);                                  \
  }
#define TCS_TC_GEO1(NN, EE, MM)                                                        \
  if (pl.geo == 1 && pl.cg == 2 && !pl.ups && pl.N == NN && pl.epi == EE && pl.msub == MM) return max_ctas_t<NN, EE, MM, 2, 1>(pl, out);
  if (pl.geo == 1 && pl.cg == 2 && pl.ups && pl.epi == EPI_PADDED && pl.N == 96 && pl.msub == 2) return max_ctas_t<96, EPI_PADDED, 2, 2, 1, 1>(pl, out);
  if (pl.geo == 1 && pl.cg == 2 && pl.ups && pl.epi == EPI_PADDED && pl.N == 192 && pl.msub == 1) return max_ctas_t<192, EPI_PADDED, 1, 2, 1, 1>(pl, out);
  TCS_TC_CASE(96, EPI_RAW_STATS, 2)
  TCS_TC_CASE(96, EPI_PADDED, 2)
  TCS_TC_CASE(96, EPI_PLAIN, 2)
  TCS_TC_CASE(96, EPI_GN_FUSED, 2)
  TCS_TC_CASE(192, EPI_RAW_STATS, 1)
  TCS_TC_CASE(192, EPI_PADDED, 1)
  TCS_TC_CASE(192, EPI_PLAIN, 1)
  TCS_TC_CASE(192, EPI_GN_FUSED, 1)
  TCS_TC_CASE(16, EPI_EPS, 2)
  TCS_TC_GEO1(96, EPI_RAW_STATS, 2)
  TCS_TC_GEO1(96, EPI_PADDED, 2)
  TCS_TC_GEO1(96, EPI_GN_FUSED, 2)
  TCS_TC_GEO1(192, EPI_RAW_STATS, 1)
  TCS_TC_GEO1(192, EPI_PADDED, 1)
  TCS_TC_GEO1(192, EPI_GN_FUSED, 1)
#undef TCS_TC_CASE
#undef TCS_TC_GEO1
  return fail(TCS_ERR_UNSUPPORTED, "conv_tc: no kernel instance for this (N, epilogue, msub)");
}

int conv_tc_launch(const ConvTcPlan& pl, cudaStream_t st) {
  if (!pl.valid) return fail(TCS_ERR_STATE, "conv_tc_launch: plan not built");
#define TCS_TC_CASE(NN, EE, MM)                                                        \
  if (pl.geo == 0 && pl.N == NN && pl.epi == EE && pl.msub == MM) {                     \
    if (pl.cg == 2) { if constexpr (NN >= 96 || EE == EPI_EPS) return launch_t<NN, EE, MM, 2, 0>(pl, st); } \
    else return launch_t<NN, EE, MM, 1, 0>(pl, st);                                     \
  }
#define TCS_TC_GEO1(NN, EE, MM)                                                        \
  if (pl.geo == 1 && pl.cg == 2 && !pl.ups && pl.N == NN && pl.epi == EE && pl.msub == MM) return launch_t<NN, EE, MM, 2, 1>(pl, st);
  if (pl.geo == 1 && pl.cg == 2 && pl.ups && pl.epi == EPI_PADDED && pl.N == 96 && pl.msub == 2) return launch_t<96, EPI_PADDED, 2, 2, 1, 1>(pl, st);
  if (pl.geo == 1 && pl.cg == 2 && pl.ups && pl.epi == EPI_PADDED && pl.N == 192 && pl.msub == 1) return launch_t<192, EPI_PADDED, 1, 2, 1, 1>(pl, st);
  TCS_TC_CASE(96, EPI_RAW_STATS, 2)
  TCS_TC_CASE(96, EPI_PADDED, 2)
  TCS_TC_CASE(96, EPI_PLAIN, 2)
  TCS_TC_CASE(96, EPI_GN_FUSED, 2)
  TCS_TC_CASE(192, EPI_RAW_STATS, 1)
  TCS_TC_CASE(192, EPI_PADDED, 1)
  TCS_TC_CASE(192, EPI_PLAIN, 1)
  TCS_TC_CASE(192, EPI_GN_FUSED, 1)
  TCS_TC_CASE(16, EPI_EPS, 2)
  TCS_TC_GEO1(96, EPI_RAW_STATS, 2)
  TCS_TC_GEO1(96, EPI_PADDED, 2)
  TCS_TC_GEO1(96, EPI_GN_FUSED, 2)
  TCS_TC_GEO1(192, EPI_RAW_STATS, 1)
  TCS_TC_GEO1(192, EPI_PADDED, 1)
  TCS_TC_GEO1(192, EPI_GN_FUSED, 1)
#undef TCS_TC_CASE
#undef TCS_TC_GEO1
  return fail(TCS_ERR_UNSUPPORTED, "conv_tc_launch: no kernel instance for this (N, epilogue, msub)");
}

int conv_tc_make_plan(ConvTcPlan* plan, const ConvGeom& g, const void* src0, const void* src1,
                      const __nv_bfloat16* wpacked, int epi, const EpiArgs& ea, int sm_count, const void* lo0,
                      const void* lo1) {
  PFN_encodeTiled encode = get_encode();
  if (!encode) return fail(TCS_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  if (g.W != 64 && g.W != 32 && g.W != 16) return fail(TCS_ERR_UNSUPPORTED, "conv_tc: output width must be 64/32/16");
  if ((g.H * g.W) % 128) return fail(TCS_ERR_UNSUPPORTED, "conv_tc: image must be a multiple of 128 pixels");
  ConvTcPlan& pl = *plan;
  pl = ConvTcPlan();
  ConvTcParams& p = pl.p;
  conv_tc_tile_shape(g, epi, &pl.N, &pl.cg);
  if (g.ntot % pl.N) return fail(TCS_ERR_UNSUPPORTED, "conv_tc: C_out must be a multiple of 96");
  pl.epi = epi;
  // N = 96: two 128-pixel sub-tiles per CTA tile share every weight (B) stage (half the B traffic per
  // MAC) and give each of the 8 epilogue warps a 32-row x 96-column unit; N = 192: one sub-tile, the
  // epilogue warps split its columns in halves.  Either way two accumulator sets double-buffer in TMEM.
  pl.msub = pl.N == 192 ? 1 : 2;
  if (epi == EPI_EPS && pl.cg == 2 && (g.B * (g.H / (2 * (128 / g.W)))) % 2)
    return fail(TCS_ERR_UNSUPPORTED, "conv_tc: the output conv runs as CTA pairs and needs an even number of tiles");
  if (g.H % (pl.msub * (128 / g.W))) return fail(TCS_ERR_UNSUPPORTED, "conv_tc: image height not a multiple of the tile");
  p.debug = getenv("TCS_DEBUG") ? atoi(getenv("TCS_DEBUG")) : 0;
  p.gn_inv_cnt = 1.0 / (static_cast<double>(g.H) * g.W * (pl.N / 8));
  p.exch_timeout = getenv("TCS_EXCHANGE_TIMEOUT") ? atoll(getenv("TCS_EXCHANGE_TIMEOUT")) : EXCHANGE_TIMEOUT_CYCLES;
  {
    const char* e = getenv("TCS_ISSUERS");   // 1 = a single MMA-issuing thread everywhere (A/B switch)
    p.issuers = (pl.msub == 2 && !(e && atoi(e) == 1)) ? 2 : 1;
  }
  stage_shape(g, &p.T, &p.KYG, &p.KW);
  p.H = g.H; p.W = g.W; p.Rt = 128 / g.W;
  p.stride = g.stride;
  p.pair = 0;
  p.kxn = g.kx_in_n ? 1 : 0;
  p.guidance = 0.f;
  p.WR = p.Rt * pl.msub + p.T - 1;
  p.nsrc = g.nsrc * (g.split3 ? 3 : 1);
  pl.cin[0] = g.csrc[0]; pl.cin[1] = g.csrc[g.nsrc > 1 ? 1 : 0];
  if (g.split3 && (!lo0 || (g.nsrc == 2 && !lo1))) return fail(TCS_ERR_BAD_ARGUMENT, "conv_tc: bf16x3 mode needs the lo parts of its sources");
  if (g.split3 && epi != EPI_RAW_STATS) return fail(TCS_ERR_UNSUPPORTED, "conv_tc: bf16x3 mode writes fp32 (EPI_RAW_STATS) only");
  p.ntot = g.ntot;
  p.tiles_per_img = g.H / (p.Rt * pl.msub);
  p.n_mtiles = g.B * p.tiles_per_img;
  p.n_ntiles = g.ntot / pl.N;
  p.kstages = conv_tc_kstages(g);
  p.a_bytes = static_cast<uint32_t>(p.WR) * g.W * ROWB;
  p.stage_bytes = (p.a_bytes + p.T * (pl.N / pl.cg) * ROWB + 1023u) & ~1023u;
  const size_t budget = 227 * 1024 - 2048 - 1024 - EPI_SLAB_BYTES - EPI_BIAS_BYTES - EPI_FUSED_BYTES;
  p.nstage = static_cast<int>(budget / p.stage_bytes);
  if (p.nstage > MAX_STAGES) p.nstage = MAX_STAGES;
  pl.geo = (pl.cg == 2) ? conv_tc_geo(g, epi) : 0;
  if (!pl.geo && p.nstage < 2) return fail(TCS_ERR_UNSUPPORTED, "conv_tc: stage does not fit shared memory twice");
  pl.smem = static_cast<size_t>(p.nstage) * p.stage_bytes + 1024 + EPI_SLAB_BYTES + EPI_BIAS_BYTES + EPI_FUSED_BYTES;
  p.geo = pl.geo;
  p.P = p.tiles_x = p.a_stages = p.tb = 0;
  p.a_load_bytes = 0;
  p.ups = p.l_stages = 0;
  p.l_bytes = p.l_load_bytes = 0;
  if (pl.geo) {
    // tap-shift geometry: CTA tile = 16 image rows x 8 MSUB pixels; one (16 + 2) x (8 MSUB + 2) pixel window per
    // 64-channel block in a ring of its own, the weights in stages of tb taps (three ky taps of one kx, or single taps
    // when three such stages would not fit: N = 192)
    if (g.W % (8 * pl.msub) || g.H % 16) return fail(TCS_ERR_UNSUPPORTED, "conv_tc: image is not a multiple of the 16 x 8 tile");
    const int NB = pl.N / pl.cg;
    p.P = 8 * pl.msub + 2;
    p.tiles_x = g.W / (8 * pl.msub);
    p.WR = 18;
    p.tiles_per_img = (g.H / 16) * p.tiles_x;
    p.n_mtiles = g.B * p.tiles_per_img;
    p.a_load_bytes = static_cast<uint32_t>(p.WR) * p.P * ROWB;
    p.a_bytes = (p.a_load_bytes + 1023u) & ~1023u;
    p.a_stages = 2;
    if (g.ups) {   // low-resolution windows: (8 + 2) rows x (4 MSUB + 2) pixels x 64 channels
      p.ups = pl.ups = 1;
      p.l_stages = 2;
      p.l_load_bytes = 10u * static_cast<uint32_t>(p.P / 2 + 1) * ROWB;
      p.l_bytes = (p.l_load_bytes + 1023u) & ~1023u;
    }
    const size_t slab_bytes = g.ups ? EPI_SLAB_BYTES / SLAB_BUFS : EPI_SLAB_BYTES;   // UPS: single-buffered output staging
    const size_t budget1 = TC_SMEM_MAX - 1024 - slab_bytes - bias_bytes_of(g.ntot) - EPI_FUSED_BYTES -
                           static_cast<size_t>(p.l_stages) * p.l_bytes;
    // what to do with the 32 KB (measured, profiles/r2_layer_speed_fused_upsample.txt): us1_conv (N = 96, a 64- and a
    // 32-channel block per tile) gains 2 % from a third window stage (2 weight stages left), us2_conv (N = 192) gains 5 %
    // from a third weight stage instead
    const bool want3 = getenv("TCS_UPS_A_STAGES") ? atoi(getenv("TCS_UPS_A_STAGES")) == 3 : pl.msub == 2;
    if (g.ups && want3 && budget1 >= 3 * static_cast<size_t>(p.a_bytes) + 2 * static_cast<size_t>(3u * NB * ROWB))
      p.a_stages = 3;
    const size_t rest = budget1 - static_cast<size_t>(p.a_stages) * p.a_bytes;
    p.tb = (rest / (3u * NB * ROWB) >= (g.ups ? 2u : 3u)) ? 3 : 1;   // (ups: two 3-tap stages beat seven 1-tap stages)
    if (getenv("TCS_TB")) p.tb = atoi(getenv("TCS_TB")) == 3 ? 3 : 1;
    p.stage_bytes = (static_cast<uint32_t>(p.tb) * NB * ROWB + 1023u) & ~1023u;
    p.nstage = static_cast<int>(rest / p.stage_bytes);
    if (p.nstage > MAX_STAGES) p.nstage = MAX_STAGES;
    if (getenv("TCS_NSTAGE") && atoi(getenv("TCS_NSTAGE")) < p.nstage) p.nstage = atoi(getenv("TCS_NSTAGE"));   // experiment
    if (getenv("TCS_PLAN_LOG")) fprintf(stderr, "[conv_tc plan] H=%d N=%d K=%d ups=%d tb=%d nstage=%d stage_bytes=%u a_bytes=%u l_bytes=%u\n", g.H, pl.N, p.kstages, p.ups, p.tb, p.nstage, p.stage_bytes, p.a_bytes, p.l_bytes);
    if (p.nstage < 2) return fail(TCS_ERR_UNSUPPORTED, "conv_tc: weight stage does not fit shared memory twice");
    pl.smem = static_cast<size_t>(p.a_stages) * p.a_bytes + static_cast<size_t>(p.l_stages) * p.l_bytes +
              static_cast<size_t>(p.nstage) * p.stage_bytes + 1024 + slab_bytes + bias_bytes_of(g.ntot) + EPI_FUSED_BYTES;
  }
  if (g.ups && !(pl.geo == 1 && pl.cg == 2 && epi == EPI_PADDED && g.nsrc == 1 && !g.split3))
    return fail(TCS_ERR_UNSUPPORTED, "conv_tc: the fused upsample needs a 3x3 stride-1 layer with one padded bf16 source and a padded output");
  p.epi = ea;
  TCS_CHECK(conv_tc_max_ctas(pl, &pl.max_ctas));
  if (getenv("TCS_MAX_CTAS")) pl.max_ctas = atoi(getenv("TCS_MAX_CTAS"));   // test hook: pretend part of the device is taken
  pl.coop_cluster = pl.cg == 2 && epi == EPI_GN_FUSED && coop_cluster_supported();
  pl.grid = conv_tc_grid(pl, g.B, sm_count);
  if (epi == EPI_GN_FUSED && (p.n_ntiles != 1 || pl.grid < p.tiles_per_img))
    return fail(TCS_ERR_UNSUPPORTED,
                "conv_tc: fused GroupNorm needs one N tile and a whole image group (" + std::to_string(p.tiles_per_img) +
                    " CTAs) resident at once; the device can hold " + std::to_string(pl.max_ctas));

  // tensor maps: [src0, src1] or, in bf16x3 mode, [hi0, lo0, hi1, lo1]; physical K segments select among them
  const void* srcs[4] = {src0, src1, src0, src1};
  int lsrc[4] = {0, 1, 0, 1};            // logical source of each map
  if (g.split3) {
    srcs[0] = src0; srcs[1] = lo0; srcs[2] = src1; srcs[3] = lo1;
    lsrc[0] = lsrc[1] = 0; lsrc[2] = lsrc[3] = 1;
  }
  for (int ps = 0; ps < 6; ++ps) {
    const int ls = g.split3 ? ps / 3 : ps;                 // logical source of this K segment
    const int li = ls < g.nsrc ? ls : 0;
    const int conv_pad = (g.ksize == 1) ? 0 : 1;           // halo 1, conv pad: 3x3 -> 1, 4x4/s2 -> 1, 1x1 -> 0
    p.base_off[ps] = g.in_pad[li] - conv_pad;
    if (p.base_off[ps] < 0) return fail(TCS_ERR_BAD_ARGUMENT, "conv_tc: a 3x3/4x4 conv needs a padded source");
    p.cblk[ps] = (g.csrc[li] + KB - 1) / KB;
    p.ctail[ps] = (g.csrc[li] % KB) ? 1 : 0;
    if (g.csrc[li] % 32) return fail(TCS_ERR_UNSUPPORTED, "conv_tc: source channels must be a multiple of 32");
    p.msel[ps] = g.split3 ? 2 * li + (ps % 3 == 2 ? 1 : 0) : li;   // [a_hi, a_hi, a_lo]
  }
  for (int s = 0; s < 4; ++s) {
    int si = lsrc[s] < g.nsrc ? lsrc[s] : 0;  // unused maps mirror the first source
    if (!srcs[s] || lsrc[s] >= g.nsrc) { srcs[s] = srcs[0]; si = 0; }
    const int pad = g.in_pad[si];
    const int Hin = g.H * g.stride + 2 * pad, Win = g.W * g.stride + 2 * pad;
    const cuuint64_t C = g.csrc[si];
    cuuint64_t dims[4] = {C, static_cast<cuuint64_t>(Win), static_cast<cuuint64_t>(Hin), static_cast<cuuint64_t>(g.B)};
    cuuint64_t strides[3] = {C * 2, C * 2 * Win, C * 2 * Win * Hin};
    cuuint32_t box[4] = {KB, static_cast<cuuint32_t>(g.W * g.stride), static_cast<cuuint32_t>(p.WR * g.stride), 1};
    cuuint32_t estr[4] = {1, static_cast<cuuint32_t>(g.stride), static_cast<cuuint32_t>(g.stride), 1};
    if (pl.geo) { box[1] = static_cast<cuuint32_t>(p.P); box[2] = static_cast<cuuint32_t>(p.WR); }
    if (pl.ups) {   // the half-resolution padded tensor, boxes of (8 + 2) x (4 MSUB + 2) pixels
      dims[1] = static_cast<cuuint64_t>(g.W / 2 + 2); dims[2] = static_cast<cuuint64_t>(g.H / 2 + 2);
      strides[1] = C * 2 * dims[1]; strides[2] = strides[1] * dims[2];
      box[1] = static_cast<cuuint32_t>(p.P / 2 + 1); box[2] = 10;
    }
    CUresult r = encode(&pl.mapA[s], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(srcs[s]), dims, strides,
                        box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, pl.ups ? CU_TENSOR_MAP_SWIZZLE_NONE : CU_TENSOR_MAP_SWIZZLE_128B,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(TCS_ERR_CUDA, "cuTensorMapEncodeTiled(A) failed: " + std::to_string(r));
  }
  {
    // the packed weights ARE the swizzled shared-memory image: plain (unswizzled) 512-byte rows
    const uint32_t stage_b = static_cast<uint32_t>(p.T) * (pl.N / pl.cg) * ROWB;   // bytes per packed K stage and CTA
    if (stage_b % 512) return fail(TCS_ERR_UNSUPPORTED, "conv_tc: weight stage is not a multiple of 512 bytes");
    p.b_rows = static_cast<int>(stage_b / 512);
    const cuuint64_t total_rows = static_cast<cuuint64_t>(p.kstages) * p.n_ntiles * pl.cg * p.b_rows;
    if (pl.geo) p.b_rows = p.b_rows * p.tb / 3;     // rows one load takes: tb of the three ky taps of a packed stage
    cuuint64_t dims[2] = {256, total_rows};
    cuuint64_t strides[1] = {512};
    cuuint32_t box[2] = {256, static_cast<cuuint32_t>(p.b_rows)};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = encode(&pl.mapW, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<__nv_bfloat16*>(wpacked), dims,
                        strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(TCS_ERR_CUDA, "cuTensorMapEncodeTiled(W) failed: " + std::to_string(r));
  }
  pl.mapO = pl.mapW;
  pl.mapO1 = pl.mapW;
  if (epi == EPI_PLAIN) {   // bf16 [M = B*H*W, ldo] output, 32-row x 32-channel boxes
    const cuuint64_t C = static_cast<cuuint64_t>(ea.ldo);
    cuuint64_t dims[2] = {C, static_cast<cuuint64_t>(g.B) * g.H * g.W};
    cuuint64_t strides[1] = {C * 2};
    cuuint32_t box[2] = {BLK, 32};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = encode(&pl.mapO, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, ea.out, dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(TCS_ERR_CUDA, "cuTensorMapEncodeTiled(O plain) failed: " + std::to_string(r));
  }
  if (epi == EPI_GN_FUSED || epi == EPI_PADDED) {   // bf16 padded output, 32-pixel (16 for 16-pixel rows) x 32-channel boxes
    const cuuint64_t C = static_cast<cuuint64_t>(ea.ldo);
    cuuint64_t dims[4] = {C, static_cast<cuuint64_t>(g.W + 2), static_cast<cuuint64_t>(g.H + 2), static_cast<cuuint64_t>(g.B)};
    cuuint64_t strides[3] = {C * 2, C * 2 * (g.W + 2), C * 2 * (g.W + 2) * (g.H + 2)};
    cuuint32_t box[4] = {BLK, static_cast<cuuint32_t>(g.W >= 32 ? 32 : 16), 1, 1};
    if (pl.geo) { box[1] = 8; box[2] = 4; }       // a warp's 32 rows = 4 image rows x 8 pixels
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = encode(&pl.mapO, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, ea.out, dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, BLK == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(TCS_ERR_CUDA, "cuTensorMapEncodeTiled(O padded) failed: " + std::to_string(r));
    if (pl.geo) {
      box[2] = 1;
      r = encode(&pl.mapO1, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, ea.out, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                 CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) return fail(TCS_ERR_CUDA, "cuTensorMapEncodeTiled(O padded, one row) failed: " + std::to_string(r));
    }
  }
  pl.valid = true;
  return TCS_OK;
}

}  // namespace tcs
