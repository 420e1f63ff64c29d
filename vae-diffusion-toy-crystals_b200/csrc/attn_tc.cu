// attn_tc.cu — SelfAttention2d (sde_score_model.py:136-167) of a 16x16x192 image as ONE tcgen05 kernel:
//   GroupNorm(8 groups) -> qkv 1x1 conv -> per head softmax(q k^T / sqrt(48)) v -> proj 1x1 conv -> + x
// q, k, v, the scores and the attention output never leave the SM (shared / tensor memory).  It replaces four
// launches of round 1 (gn_image16, conv_tc<attn.qkv>, an mma.sync attention kernel, conv_tc<attn.proj>).
//
// Work split: an image (256 tokens) is a CLUSTER OF TWO CTAs, each owning 128 tokens = the 128 TMEM lanes = one M tile.
// Every CTA projects q, k, v of its own tokens and pushes its 128 k / v rows into the peer's shared memory (one bulk
// shared::cluster copy per operand, completing on the peer's mbarrier), so that each CTA holds all 256 keys of the
// current head.  All MMAs are cta_group::1 (M = 128):
//   qkv_h [128 x 144] = Xn [128 x 192] . W_h^T        A, B shared memory (K-major SWIZZLE_128B), per head h
//   S     [128 x 256] = Q'_h [128 x 48] . K_h^T       A = Q' in TENSOR MEMORY (bf16 packed, tcgen05.st), Q' = q log2e/sqrt(48)
//   O_h   [128 x  64] = P [128 x 256] . V_h           A = P (fp16) in tensor memory, written IN PLACE over the S columns;
//                                                     B = V rows (keys) x 64 (fp16: 48 values, a 1, zeros) -> MN-major
//                                                     descriptor; column 48 of O_h is the softmax denominator
//   Y     [128 x 192] = O [128 x 192] . Wproj^T       A = normalised O of all heads (shared memory)
// TMEM columns: [0,256) S / P / Y, [256,400) qkv_h, [400,424) Q' (packed), [424,488) O_h (48 columns + the row sums).
// Shared memory (214 KB): Xn 48 K | weights of the head 54 K (bulk-copied, pre-swizzled images; Wproj reuses this and the
// dead Xn region) | K 32 K | V 32 K (128-byte rows, 48 of 64 elements used) | O 48 K.
// Threads: warp 0 = control (one lane issues the bulk copies and every MMA), warps 1-8 = workers: warp w owns TMEM lane
// quarter w % 4 (32 tokens) and column half (w - 1) / 4 of whatever is being read, so a softmax row is shared by two
// threads (the row maximum is combined through shared memory, the row sum comes out of the P V product).
// Protocol: mbarriers only (struct AttnBars); the control lane issues the next head's projection right after S_h and the
// P V product chunk by chunk behind the softmax; the workers convert the next head's q, k / v while the tensor core works.
// The one cluster-wide barrier per image is the GroupNorm statistics exchange.
// The building blocks (A operand in tensor memory, MN-major partial atom, DSMEM-written operands, 1-D bulk copies)
// were probed on B200 first: tools/umma_attn_probe.cu, profiles/r2_attn_probe.txt.
#include <cooperative_groups.h>

#include <cstdlib>
#include <cstring>
#include <mutex>

#include "attn_tc.cuh"
#include "tc_ptx.cuh"

namespace cg = cooperative_groups;

namespace tcs {
namespace {

constexpr int AT_THREADS = 288;
constexpr int AT_TOK = 128;
constexpr int AT_PIMG = 18 * 18 * 192;                 // elements of a padded image
constexpr uint32_t XN_OFF = 0, W_OFF = 49152, K_OFF = 104448, V_OFF = 137216, O_OFF = 169984, AT_SMEM = 219136;
constexpr uint32_t KBLK = 16384;                       // a 128-row x 64-channel K block of an A operand
constexpr uint32_t WH_KB = 144 * 128, WH_BYTES = 3 * WH_KB;       // per-head q|k|v weights
constexpr uint32_t WP_KB = 192 * 128, WP_BYTES = 3 * WP_KB;       // projection weights
constexpr uint32_t R_OFF = K_OFF;                     // epilogue staging rows [128][384 B] over the idle K / V regions
constexpr uint32_t S_COL = 0, QKV_COL = 256, Q_COL = 400, O_COL = 424;
constexpr float QSCALE = 0.14433756729740643f * 1.4426950408889634f;   // log2(e) / sqrt(48)
static_assert(W_OFF % 1024 == 0 && K_OFF % 1024 == 0 && V_OFF % 1024 == 0 && O_OFF % 1024 == 0, "swizzle atoms");
static_assert(W_OFF + WH_BYTES == K_OFF && 2 * WP_KB <= WH_BYTES && WP_KB <= W_OFF, "weight regions");

__host__ __device__ inline uint32_t sw128(uint32_t row, uint32_t ch) { return row * 128 + ((ch ^ (row & 7)) << 4); }

__device__ __forceinline__ uint32_t pack2(float a, float b) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ void unpack8(const uint4& u, float* f) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 t = __bfloat1622float2(h[i]);
    f[2 * i] = t.x; f[2 * i + 1] = t.y;
  }
}
__device__ __forceinline__ uint4 pack8(const float* f) {
  return make_uint4(pack2(f[0], f[1]), pack2(f[2], f[3]), pack2(f[4], f[5]), pack2(f[6], f[7]));
}
// fp16 pair (a in the low half), round to nearest, saturating to the largest finite value
__device__ __forceinline__ uint32_t pack2_f16(float a, float b) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}
__device__ __forceinline__ uint4 pack8_f16(const float* f) {
  return make_uint4(pack2_f16(f[0], f[1]), pack2_f16(f[2], f[3]), pack2_f16(f[4], f[5]), pack2_f16(f[6], f[7]));
}
// two base-2 exponentials per MUFU operation
__device__ __forceinline__ uint32_t ex2_f16x2(uint32_t x) {
  uint32_t y;
  asm("ex2.approx.f16x2 %0, %1;" : "=r"(y) : "r"(x));
  return y;
}
// instruction descriptor for kind::f16 with fp16 A and B (the P V product: P and V are stored as fp16)
__host__ __device__ constexpr uint32_t make_idesc_f16(int M, int N) {
  return (1u << 4) | (static_cast<uint32_t>(N >> 3) << 17) | (static_cast<uint32_t>(M >> 4) << 24);
}
__device__ __forceinline__ void worker_bar() { asm volatile("bar.sync 1, 256;" ::: "memory"); }
__device__ __forceinline__ int halo_wrap16(int v) { return v == 0 ? 16 : (v == 15 ? -16 : 0); }

// ---- cluster helpers ------------------------------------------------------------------------------------------------
// arrive on the PEER CTA's copy of a barrier; relaxed: it only says "my MMAs have finished reading your rows"
__device__ __forceinline__ void mbar_arrive_peer(uint32_t bar, uint32_t peer) {
  asm volatile(
      "{\n\t.reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [ra];\n\t}" ::"r"(bar), "r"(peer) : "memory");
}
// bulk copy own shared memory -> the same offset in the peer CTA, completing (bytes) on the peer's barrier
__device__ __forceinline__ void bulk_push_to_peer(uint32_t addr, uint32_t bytes, uint32_t bar, uint32_t peer) {
  asm volatile(
      "{\n\t.reg .b32 rd, rb;\n\t"
      "mapa.shared::cluster.u32 rd, %0, %3;\n\t"
      "mapa.shared::cluster.u32 rb, %2, %3;\n\t"
      "cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [rd], [%0], %1, [rb];\n\t}"
      ::"r"(addr), "r"(bytes), "r"(bar), "r"(peer) : "memory");
}

__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, uint32_t src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(map)), "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
// tensor maps of the padded [B,18,18,192] bf16 input / output (SWIZZLE_128B, 64-channel boxes)
struct AttnTcMaps {
  CUtensorMap x;         // box 64 ch x 16 px x 8 rows: one CTA's rows of a K block
  CUtensorMap out;       // the same box over the output tensor
  CUtensorMap out_row;   // box 64 ch x 16 px x 1 row (the wrapped halo rows)
};

struct AttnBars {
  uint64_t w, qkv, s, o, y;          // weights landed / qkv_h, S, O_h, Y accumulators complete (tcgen05.commit)
  uint64_t klocal, vlocal;           // this CTA's workers have stored Q' + their K rows / their V rows (8 warp arrivals)
  uint64_t kfull, vfull;             // the peer's 128 K / V rows have landed here (bulk push, 16 KB each)
  uint64_t kfree, vfree;             // the peer's MMAs are done with the rows this CTA pushed (remote arrive)
  uint64_t odone;                    // all heads' attention outputs are in shared memory (8 warp arrivals)
  uint64_t resid;                    // this image's input rows (residual) have landed in the staging rows (3 TMA boxes)
  uint64_t xrows;                    // the next image's raw input rows have landed in the O region (8 bulk copies)
  uint64_t pready[4];                // softmax chunk i of every worker warp is in tensor memory (8 warp arrivals)
};

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(AT_THREADS, 1) attn_block_tc_kernel(const __grid_constant__ AttnTcMaps maps, const AttnTcParams p) {
  extern __shared__ uint8_t at_raw[];
  __shared__ AttnBars bars;
  __shared__ uint32_t tmem_slot;
  __shared__ float s_part[AT_THREADS][2];
  __shared__ float s_mine[16], s_peer[16];
  __shared__ float s_mean[8], s_rstd[8];
  __shared__ float s_max[2][AT_TOK];
  __shared__ float s_bqkv[576], s_bproj[192], s_gamma[192], s_beta[192];

  cg::cluster_group cluster = cg::this_cluster();
  const uint32_t rank = cluster.block_rank(), peer = rank ^ 1u;
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);   // warp-uniform role dispatch
  const bool ctrl = warp == 0;
  uint8_t* sm = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(at_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  const uint32_t sb = ptx::smem_u32(sm);
  float* peer_part = cluster.map_shared_rank(&s_peer[0], peer);
  const uint32_t b_w = ptx::smem_u32(&bars.w), b_qkv = ptx::smem_u32(&bars.qkv), b_s = ptx::smem_u32(&bars.s),
                 b_o = ptx::smem_u32(&bars.o), b_y = ptx::smem_u32(&bars.y), b_kl = ptx::smem_u32(&bars.klocal),
                 b_vl = ptx::smem_u32(&bars.vlocal), b_kf = ptx::smem_u32(&bars.kfull), b_vf = ptx::smem_u32(&bars.vfull),
                 b_kfree = ptx::smem_u32(&bars.kfree), b_vfree = ptx::smem_u32(&bars.vfree),
                 b_od = ptx::smem_u32(&bars.odone), b_p0 = ptx::smem_u32(&bars.pready[0]), b_x = ptx::smem_u32(&bars.xrows), b_r = ptx::smem_u32(&bars.resid);

  for (int i = tid; i < 576; i += AT_THREADS) s_bqkv[i] = p.bias_qkv[i];
  for (int i = tid; i < 192; i += AT_THREADS) { s_bproj[i] = p.bias_proj[i]; s_gamma[i] = p.gamma[i]; s_beta[i] = p.beta[i]; }
  if (tid == 0) {
    for (uint32_t b : {b_w, b_qkv, b_s, b_o, b_y, b_kf, b_vf, b_kfree, b_vfree, b_x, b_r}) ptx::mbar_init(b, 1);
    for (uint32_t b : {b_kl, b_vl, b_od}) ptx::mbar_init(b, 8);
    for (int i = 0; i < 4; ++i) ptx::mbar_init(b_p0 + 8 * i, 8);
    ptx::fence_barrier_init();
  }
  if (tid == 32) { ptx::prefetch_tmap(&maps.x); ptx::prefetch_tmap(&maps.out); ptx::prefetch_tmap(&maps.out_row); }
  if (ctrl) ptx::tmem_alloc_512(ptx::smem_u32(&tmem_slot));
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem = tmem_slot;
  cluster.sync();   // the peer is running and its barriers are initialised: its shared memory may be written from here on

  const int ncl = gridDim.x >> 1, cl = blockIdx.x >> 1;
  // phase parities, one set per waiting role (control lane / workers); every wait flips its own bit
  uint32_t ph_w = 0, ph_qkv = 0, ph_s = 0, ph_o = 0, ph_y = 0, ph_kl = 0, ph_vl = 0, ph_kf = 0, ph_vf = 0, ph_kfree = 0,
           ph_vfree = 0, ph_od = 0, ph_p = 0, ph_x = 0, ph_r = 0;
  if (ctrl && lane == 0 && cl < p.B) {
    ptx::mbar_expect_tx(b_w, WH_BYTES);
    ptx::bulk_load_1d(sb + W_OFF, p.wpack, WH_BYTES, b_w);
    // the peer's 128 K / V rows of a head land here: each phase is armed as soon as the previous one has completed, i.e.
    // always before this CTA lets the peer push again (kfree / vfree, or the per-image cluster barrier)
    ptx::mbar_expect_tx(b_kf, 16384);
    ptx::mbar_expect_tx(b_vf, 16384);
  }
  // worker coordinates (meaningless for the control warp)
  const int wq = warp & 3, hf = (warp - 1) >> 2;
  const int row = wq * 32 + lane;                    // token inside this CTA = TMEM lane
  const int gt = static_cast<int>(rank) * AT_TOK + row;   // token inside the image = key index
  const int wt = tid - 32;                           // worker thread index 0..255
  const uint32_t lane_addr = tmem + (static_cast<uint32_t>(wq * 32) << 16);
  // phase-0 coordinates: thread = (16-byte channel chunk, token lane)
  const int c0 = tid % 24, tl = tid / 24;

  // raw x of this CTA's 8 image rows of image `im` -> the O region as plain [token][384 B] rows: one 6144-byte bulk copy
  // per image row (16 pixels are contiguous in the padded tensor); phase 0 normalises them into the Xn slots
  auto fetch_x = [&](int im) {
    const __nv_bfloat16* src = p.x + static_cast<size_t>(im) * AT_PIMG;
    ptx::mbar_expect_tx(b_x, 8 * 6144);
#pragma unroll
    for (int r = 0; r < 8; ++r)
      ptx::bulk_load_1d(sb + O_OFF + r * 6144, src + ((static_cast<int>(rank) * 8 + r + 1) * 18 + 1) * 192, 6144, b_x);
  };
  if (ctrl && lane == 0 && cl < p.B) fetch_x(cl);

  for (int img = cl; img < p.B; img += ncl) {
    __nv_bfloat16* ob = p.out + static_cast<size_t>(img) * AT_PIMG;
    float* dbg = (p.dbg && img == 0) ? p.dbg : nullptr;
    // ---- phase 0 (all threads): GroupNorm statistics over both CTAs' halves, Xn normalised in place -----------------
    {
      uint4 v[11];
      ptx::mbar_wait(b_x, ph_x); ph_x ^= 1;   // the raw rows (fetch_x in the previous image's tail)
#pragma unroll
      for (int k = 0; k < 11; ++k) {
        const int tok = tl + 12 * k;
        if (tok < AT_TOK) v[k] = *reinterpret_cast<const uint4*>(sm + O_OFF + tok * 384 + c0 * 16);
      }
      float s = 0.f, q = 0.f;
#pragma unroll
      for (int k = 0; k < 11; ++k) {
        if (tl + 12 * k < AT_TOK) {
          float f[8];
          unpack8(v[k], f);
#pragma unroll
          for (int j = 0; j < 8; ++j) { s += f[j]; q += f[j] * f[j]; }
        }
      }
      s_part[tid][0] = s; s_part[tid][1] = q;
      __syncthreads();
      if (tid < 64) {   // fixed-order combine (run-to-run bit-identical): 4 lanes x 9 partials per (group, sum | sum of squares)
        const int pair = tid >> 2, part = tid & 3, g = pair >> 1, which = pair & 1;
        float a = 0.f;
#pragma unroll
        for (int j = 0; j < 9; ++j) {
          const int idx = part * 9 + j;
          a += s_part[(idx / 3) * 24 + g * 3 + idx % 3][which];
        }
        a += __shfl_xor_sync(0xffffffffu, a, 1);
        a += __shfl_xor_sync(0xffffffffu, a, 2);
        if (part == 0) { s_mine[pair] = a; peer_part[pair] = a; }
      }
      cluster.sync();   // also: both CTAs have finished the previous image (no stale traffic into reused buffers)
      if (tid < 8) {
        const float sa = rank == 0 ? s_mine[2 * tid] : s_peer[2 * tid], sb2 = rank == 0 ? s_peer[2 * tid] : s_mine[2 * tid];
        const float qa = rank == 0 ? s_mine[2 * tid + 1] : s_peer[2 * tid + 1], qb = rank == 0 ? s_peer[2 * tid + 1] : s_mine[2 * tid + 1];
        const double inv = 1.0 / (256.0 * 24.0);
        const double mean = (static_cast<double>(sa) + static_cast<double>(sb2)) * inv;
        double var = (static_cast<double>(qa) + static_cast<double>(qb)) * inv - mean * mean;
        var = var < 0.0 ? 0.0 : var;
        s_mean[tid] = static_cast<float>(mean);
        s_rstd[tid] = rsqrtf(static_cast<float>(var) + GN_EPS);
      }
      __syncthreads();
      const int g = c0 / 3;
      const float mean = s_mean[g], rstd = s_rstd[g];
      float gm[8], bt[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) { gm[j] = s_gamma[c0 * 8 + j] * rstd; bt[j] = s_beta[c0 * 8 + j] - mean * gm[j]; }
      // (x - mean) rstd gamma + beta == x (rstd gamma) + (beta - mean rstd gamma)
#pragma unroll
      for (int k = 0; k < 11; ++k) {
        const int tok = tl + 12 * k;
        if (tok < AT_TOK) {
          float f[8];
          unpack8(v[k], f);
#pragma unroll
          for (int j = 0; j < 8; ++j) f[j] = fmaf(f[j], gm[j], bt[j]);
          const uint4 u = pack8(f);
          *reinterpret_cast<uint4*>(sm + XN_OFF + (c0 >> 3) * KBLK + sw128(tok, c0 & 7)) = u;
          if (dbg) {
            float r[8];
            unpack8(u, r);
            for (int j = 0; j < 8; ++j) dbg[ATTN_DBG_XN + (static_cast<size_t>(rank) * AT_TOK + tok) * 192 + c0 * 8 + j] = r[j];
          }
        }
      }
      ptx::fence_proxy_async();
      ptx::tc_fence_before();
      ptx::bulk_wait_read<0>();   // the previous image's output rows have left the staging rows (= the K / V regions)
      __syncthreads();
    }
    if (ctrl) {
      // ================= control lane: every MMA, the weight loads, the K / V pushes to the peer =====================
      if (lane == 0) {
        ptx::tc_fence_after();
        auto issue_qkv = [&]() {   // qkv_h [128 x 144] = Xn . W_h^T (weights of the head must have landed)
          ptx::mbar_wait(b_w, ph_w); ph_w ^= 1;
          ptx::tc_fence_after();
          const uint32_t idesc = make_idesc(128, 144);
#pragma unroll
          for (int kb = 0; kb < 3; ++kb) {
            const uint64_t ad = make_desc_sw128(sb + XN_OFF + kb * KBLK), bd = make_desc_sw128(sb + W_OFF + kb * WH_KB);
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) ptx::umma_bf16(tmem + QKV_COL, ad + 2 * ks, bd + 2 * ks, idesc, (kb | ks) ? 1u : 0u);
          }
          ptx::umma_commit(b_qkv);
        };
        auto load_weights = [&](int hn) {   // after qkv_{hn-1} has completed: head hn's weights, or the projection's
          ptx::mbar_wait(b_qkv, ph_qkv); ph_qkv ^= 1;
          if (hn < N_HEADS) {
            ptx::mbar_expect_tx(b_w, WH_BYTES);
            ptx::bulk_load_1d(sb + W_OFF, p.wpack + static_cast<size_t>(hn) * WH_BYTES, WH_BYTES, b_w);
          } else {   // Xn is dead as well: the third K block of Wproj goes there
            const uint8_t* wp = p.wpack + static_cast<size_t>(N_HEADS) * WH_BYTES;
            ptx::mbar_expect_tx(b_w, WP_BYTES);
            ptx::bulk_load_1d(sb + W_OFF, wp, 2 * WP_KB, b_w);
            ptx::bulk_load_1d(sb + XN_OFF, wp + 2 * WP_KB, WP_KB, b_w);
          }
        };
        issue_qkv();
        load_weights(1);
        for (int h = 0; h < N_HEADS; ++h) {
          // K rows (and Q' in tensor memory) of my tokens are stored: push my K rows, then S as soon as the peer's are here
          ptx::mbar_wait(b_kl, ph_kl); ph_kl ^= 1;
          if (h > 0) { ptx::mbar_wait(b_kfree, ph_kfree); ph_kfree ^= 1; }
          bulk_push_to_peer(sb + K_OFF + rank * 16384, 16384, b_kf, peer);
          ptx::mbar_wait(b_kf, ph_kf); ph_kf ^= 1;
          ptx::mbar_expect_tx(b_kf, 16384);
          ptx::tc_fence_after();
          {
            const uint32_t idesc = make_idesc(128, 256);
            const uint64_t kd = make_desc_sw128(sb + K_OFF);
#pragma unroll
            for (int ks = 0; ks < 3; ++ks) ptx::umma_bf16_ts(tmem + S_COL, tmem + Q_COL + 8 * ks, kd + 2 * ks, idesc, ks ? 1u : 0u);
            ptx::umma_commit(b_s);
          }
          ptx::mbar_wait(b_vl, ph_vl); ph_vl ^= 1;
          if (h > 0) { ptx::mbar_wait(b_vfree, ph_vfree); ph_vfree ^= 1; }
          bulk_push_to_peer(sb + V_OFF + rank * 16384, 16384, b_vf, peer);
          if (h < N_HEADS - 1) issue_qkv();   // next head's projection runs under this head's softmax (qkv_h has been read)
          ptx::mbar_wait(b_s, ph_s); ph_s ^= 1;                       // S_h complete: the peer may overwrite its K rows here
          if (h < N_HEADS - 1) mbar_arrive_peer(b_kfree, peer);
          ptx::mbar_wait(b_vf, ph_vf); ph_vf ^= 1;
          ptx::mbar_expect_tx(b_vf, 16384);
          {
            const uint32_t idesc = make_idesc_f16(128, 64) | IDESC_B_MN_MAJOR;   // columns 48..: the ones column (row sums)
#pragma unroll
            for (int i = 0; i < 4; ++i) {   // O_h += P V_h for the 64 keys of softmax chunk i, as soon as that chunk is stored
              ptx::mbar_wait(b_p0 + 8 * i, ph_p);
              ptx::tc_fence_after();
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const int ks = (j >> 1) * 8 + 2 * i + (j & 1);             // 16-key step: halves 0 / 1 hold keys 0-127 / 128-255
                const uint32_t a_col = S_COL + (j >> 1) * 128 + 16 * i + 8 * (j & 1);
                ptx::umma_bf16_ts(tmem + O_COL, tmem + a_col, make_desc_sw128_mn(sb + V_OFF + ks * 2048), idesc, (i | j) ? 1u : 0u);
              }
            }
            ph_p ^= 1;
            ptx::umma_commit(b_o);
          }
          if (h < N_HEADS - 1) load_weights(h + 2);                    // qkv_{h+1} complete -> W_{h+2} / Wproj
          ptx::mbar_wait(b_o, ph_o); ph_o ^= 1;                       // O_h complete: the S / P columns and V rows are free
          if (h < N_HEADS - 1) {
            mbar_arrive_peer(b_vfree, peer);
          } else {   // the K / V regions are idle until the next image: this image's input rows (the residual) go there, as
                     // three 64-channel boxes in the K-block layout (conflict-free for one token per lane)
            ptx::mbar_expect_tx(b_r, 3 * KBLK);
#pragma unroll
            for (int kb = 0; kb < 3; ++kb)
              ptx::tma_load_4d(sb + R_OFF + kb * KBLK, &maps.x, b_r, kb * 64, 1, 1 + 8 * static_cast<int>(rank), img);
          }
        }
        // projection
        ptx::mbar_wait(b_od, ph_od); ph_od ^= 1;
        ptx::mbar_wait(b_w, ph_w); ph_w ^= 1;
        ptx::tc_fence_after();
        {
          const uint32_t idesc = make_idesc(128, 192);
#pragma unroll
          for (int kb = 0; kb < 3; ++kb) {
            const uint64_t ad = make_desc_sw128(sb + O_OFF + kb * KBLK);
            const uint64_t bd = make_desc_sw128(kb < 2 ? sb + W_OFF + kb * WP_KB : sb + XN_OFF);
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) ptx::umma_bf16(tmem + S_COL, ad + 2 * ks, bd + 2 * ks, idesc, (kb | ks) ? 1u : 0u);
          }
          ptx::umma_commit(b_y);
        }
        ptx::mbar_wait(b_y, ph_y); ph_y ^= 1;
        if (img + ncl < p.B) {   // next image: raw rows into the O region (the projection has read it), first head's weights
          fetch_x(img + ncl);
          ptx::mbar_expect_tx(b_w, WH_BYTES);
          ptx::bulk_load_1d(sb + W_OFF, p.wpack, WH_BYTES, b_w);
        }
      }
      __syncwarp();
    } else {
      // ================= workers =====================================================================================
      // q|k|v of head hh: Q' (hf 0) -> tensor memory, K rows (hf 1) -> shared memory; then (second call) the V rows
      auto convert_qk = [&](int hh) {
        ptx::mbar_wait(b_qkv, ph_qkv); ph_qkv ^= 1;
        ptx::tc_fence_after();
        float f[48];
        const uint32_t src = lane_addr + QKV_COL + 48 * hf;
        ptx::tmem_ld32(src, f);
        ptx::tmem_ld16(src + 32, f + 32);
        ptx::tmem_ld_wait();
        const float* bsrc = s_bqkv + hf * 192 + hh * 48;
        // the K rows of the previous head were the source of a push: the peer's "S complete" also says that push has landed
        if (hh > 0) { ptx::mbar_wait(b_kfree, ph_kfree); ph_kfree ^= 1; }
#pragma unroll
        for (int j = 0; j < 6; ++j) {
          float g8[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) g8[i] = f[8 * j + i] + bsrc[8 * j + i];
          if (dbg) {
            for (int i = 0; i < 8; ++i) dbg[ATTN_DBG_QKV + static_cast<size_t>(gt) * 576 + hf * 192 + hh * 48 + j * 8 + i] = g8[i];
          }
          if (hf == 0) {
#pragma unroll
            for (int i = 0; i < 8; ++i) g8[i] *= QSCALE;
            const uint4 u = pack8(g8);
            ptx::tmem_st4(lane_addr + Q_COL + j * 4, reinterpret_cast<const uint32_t*>(&u));
          } else {
            *reinterpret_cast<uint4*>(sm + K_OFF + sw128(gt, j)) = pack8(g8);
          }
        }
        if (hf == 0) ptx::tmem_st_wait(); else ptx::fence_proxy_async();
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(b_kl);
      };
      auto convert_v = [&](int hh) {
        float f[24];
        const uint32_t src = lane_addr + QKV_COL + 96 + 24 * hf;
        ptx::tmem_ld16(src, f);
        ptx::tmem_ld8(src + 16, f + 16);
        ptx::tmem_ld_wait();
        const float* bsrc = s_bqkv + 384 + hh * 48 + 24 * hf;
        if (hh > 0) { ptx::mbar_wait(b_vfree, ph_vfree); ph_vfree ^= 1; }   // same for the V rows (the peer's O complete)
#pragma unroll
        for (int j = 0; j < 3; ++j) {
          float g8[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) g8[i] = f[8 * j + i] + bsrc[8 * j + i];
          if (dbg) {
            for (int i = 0; i < 8; ++i) dbg[ATTN_DBG_QKV + static_cast<size_t>(gt) * 576 + 384 + hh * 48 + 24 * hf + j * 8 + i] = g8[i];
          }
          *reinterpret_cast<uint4*>(sm + V_OFF + sw128(gt, 3 * hf + j)) = pack8_f16(g8);
        }
        // element 48 of every V row is 1: column 48 of P V is then the softmax denominator, summed by the tensor core over
        // exactly the fp16 P values the product uses (elements 49..63 are zero / never read back)
        *reinterpret_cast<uint4*>(sm + V_OFF + sw128(gt, 6 + hf)) = hf == 0 ? make_uint4(0x3C00u, 0u, 0u, 0u) : make_uint4(0u, 0u, 0u, 0u);
        ptx::fence_proxy_async();
        ptx::tc_fence_before();     // the qkv_h columns have been read: the control lane may issue the next projection
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(b_vl);
      };
      convert_qk(0);
      convert_v(0);
      for (int h = 0; h < N_HEADS; ++h) {
        // ---- softmax over keys [128 hf, 128 hf + 128) of row `row`; P (bf16) overwrites the first half of those columns
        ptx::mbar_wait(b_s, ph_s); ph_s ^= 1;
        ptx::tc_fence_after();
        const uint32_t sc = lane_addr + S_COL + 128 * hf;
        float m = -INFINITY;
        {   // pass 1: row maximum, two 32-column loads in flight at a time
          float sv[2][32];
#pragma unroll
          for (int i = 0; i < 4; i += 2) {
            ptx::tmem_ld32(sc + 32 * i, sv[0]);
            ptx::tmem_ld32(sc + 32 * i + 32, sv[1]);
            ptx::tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 32; ++j) m = fmaxf(m, fmaxf(sv[0][j], sv[1][j]));
          }
        }
        s_max[hf][row] = m;
        worker_bar();
        m = fmaxf(s_max[0][row], s_max[1][row]);
        {   // pass 2: P = 2^(S' - m) as fp16 pairs, chunk i + 1 loading and chunk i - 1 draining while chunk i is computed
          float sv[2][32];
          ptx::tmem_ld32(sc, sv[0]);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            ptx::tmem_ld_wait();
            if (i < 3) ptx::tmem_ld32(sc + 32 * (i + 1), sv[(i + 1) & 1]);
            uint32_t pk[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) pk[j] = ex2_f16x2(pack2_f16(sv[i & 1][2 * j] - m, sv[i & 1][2 * j + 1] - m));
            if (i > 0) {   // the previous chunk's store has had this chunk's math to complete: publish it
              ptx::tmem_st_wait();
              ptx::tc_fence_before();
              __syncwarp();
              if (lane == 0) ptx::mbar_arrive(b_p0 + 8 * (i - 1));
            }
            ptx::tmem_st16(sc + 16 * i, pk);
          }
          ptx::tmem_st_wait();
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(b_p0 + 8 * 3);
        }
        // ---- next head's Q' and K rows (S_h is complete, so Q' and this CTA's K rows may be overwritten) ---------------
        if (h < N_HEADS - 1) convert_qk(h + 1);
        // ---- O_h / l -> shared memory (A operand of the projection) ----------------------------------------------------
        ptx::mbar_wait(b_o, ph_o); ph_o ^= 1;
        ptx::tc_fence_after();
        {
          float o[24], lsum;
          ptx::tmem_ld16(lane_addr + O_COL + 24 * hf, o);
          ptx::tmem_ld8(lane_addr + O_COL + 24 * hf + 16, o + 16);
          ptx::tmem_ld1(lane_addr + O_COL + 48, &lsum);
          ptx::tmem_ld_wait();
          const float inv = 1.0f / lsum;
          if (dbg && hf == 0) dbg[ATTN_DBG_L + static_cast<size_t>(gt) * 4 + h] = lsum;
#pragma unroll
          for (int j = 0; j < 3; ++j) {
            float g8[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) g8[i] = o[8 * j + i] * inv;
            const int gc = h * 6 + 3 * hf + j;   // 16-byte chunk of the 192-channel row
            *reinterpret_cast<uint4*>(sm + O_OFF + (gc >> 3) * KBLK + sw128(row, gc & 7)) = pack8(g8);
            if (dbg) {
              for (int i = 0; i < 8; ++i) dbg[ATTN_DBG_Y + static_cast<size_t>(gt) * 192 + gc * 8 + i] = g8[i];
            }
          }
        }
        // ---- next head's V rows (O_h is complete, so the V rows may be overwritten) ------------------------------------
        if (h < N_HEADS - 1) {
          convert_v(h + 1);
        } else {
          ptx::fence_proxy_async();
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(b_od);
        }
      }
      // ---- projection epilogue: y + bias + x -> bf16, in place in the staging rows (K-block layout, SWIZZLE_128B), then
      // three TMA tensor stores (+ three for the wrapped halo row); border columns are written by their own threads -------
      const int ty = gt >> 4, tx = gt & 15;
      const long long wy = static_cast<long long>(halo_wrap16(ty)) * 18 * 192, wx = static_cast<long long>(halo_wrap16(tx)) * 192;
      __nv_bfloat16* dcol = ob + static_cast<size_t>((ty + 1) * 18 + tx + 1) * 192 + 96 * hf;
      ptx::mbar_wait(b_y, ph_y); ph_y ^= 1;
      ptx::tc_fence_after();
      ptx::mbar_wait(b_r, ph_r); ph_r ^= 1;
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        float yv[32];
        ptx::tmem_ld32(lane_addr + S_COL + 96 * hf + 32 * i, yv);
        ptx::tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int ch = 12 * hf + 4 * i + j;   // 16-byte chunk of the 192-channel row
          uint4* slot = reinterpret_cast<uint4*>(sm + R_OFF + (ch >> 3) * KBLK + sw128(row, ch & 7));
          float r[8], g8[8];
          unpack8(*slot, r);
#pragma unroll
          for (int e = 0; e < 8; ++e) g8[e] = yv[8 * j + e] + s_bproj[ch * 8 + e] + r[e];
          const uint4 u = pack8(g8);
          *slot = u;
          if (wx) {   // left / right border pixel: its copy on the opposite halo column (and the corner)
            *reinterpret_cast<uint4*>(dcol + wx + (4 * i + j) * 8) = u;
            if (wy) *reinterpret_cast<uint4*>(dcol + wx + wy + (4 * i + j) * 8) = u;
          }
        }
      }
      ptx::fence_proxy_async();
      ptx::tc_fence_before();
      worker_bar();
      if (wt == 0) {
#pragma unroll
        for (int kb = 0; kb < 3; ++kb) {
          const uint32_t src = sb + R_OFF + kb * KBLK;
          tma_store_4d(&maps.out, src, kb * 64, 1, 1 + 8 * static_cast<int>(rank), img);
          if (rank == 0) tma_store_4d(&maps.out_row, src, kb * 64, 1, 17, img);                 // image row 0 -> padded row 17
          else tma_store_4d(&maps.out_row, src + 112 * 128, kb * 64, 1, 0, img);                // image row 15 -> padded row 0
        }
        ptx::bulk_commit();
      }
    }
  }
  ptx::bulk_wait_all();
  ptx::tc_fence_before();
  cluster.sync();      // no remote arrive / push may target a CTA that has exited
  if (ctrl) ptx::tmem_dealloc_512(tmem);
}

}  // namespace

size_t attn_tc_wpack_bytes() { return static_cast<size_t>(N_HEADS) * WH_BYTES + WP_BYTES; }

void attn_tc_pack_weights(const float* qkv_w, const float* proj_w, uint8_t* out) {
  std::memset(out, 0, attn_tc_wpack_bytes());
  auto put = [](uint8_t* base, uint32_t row, int ch, float v) {   // element (row, channel ch of 64) of a K block
    const __nv_bfloat16 b = __float2bfloat16(v);
    std::memcpy(base + sw128(row, ch >> 3) + (ch & 7) * 2, &b, 2);
  };
  for (int h = 0; h < N_HEADS; ++h)
    for (int r = 0; r < 144; ++r) {
      const int kind = r / 48, d = r % 48, orow = kind * 192 + h * 48 + d;   // torch.chunk(qkv, 3) then heads of 48
      for (int ci = 0; ci < 192; ++ci)
        put(out + static_cast<size_t>(h) * WH_BYTES + (ci >> 6) * WH_KB, r, ci & 63, qkv_w[orow * 192 + ci]);
    }
  uint8_t* wp = out + static_cast<size_t>(N_HEADS) * WH_BYTES;
  for (int r = 0; r < 192; ++r)
    for (int ci = 0; ci < 192; ++ci) put(wp + (ci >> 6) * WP_KB, r, ci & 63, proj_w[r * 192 + ci]);
}

int launch_attn_block_tc(const AttnTcParams& p, int sm_count, cudaStream_t st) {
  if (p.B <= 0) return TCS_OK;
  constexpr int smem = AT_SMEM + 1024;
  // per device (function attributes and cluster occupancy belong to a device; a process may hold handles on several)
  static std::mutex mu;
  static int max_clusters_dev[64];
  static bool done_dev[64] = {};
  int dev = 0;
  TCS_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) return fail(TCS_ERR_UNSUPPORTED, "attn_tc: device ordinal out of range");
  cudaError_t attr_err = cudaSuccess;
  {
    std::lock_guard<std::mutex> lock(mu);
    if (!done_dev[dev]) {
      attr_err = cudaFuncSetAttribute(attn_block_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
      if (attr_err == cudaSuccess) {
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3(2 * (sm_count / 2)); cfg.blockDim = dim3(AT_THREADS); cfg.dynamicSmemBytes = smem;
        cudaLaunchAttribute at{};
        at.id = cudaLaunchAttributeClusterDimension;
        at.val.clusterDim.x = 2; at.val.clusterDim.y = 1; at.val.clusterDim.z = 1;
        cfg.attrs = &at; cfg.numAttrs = 1;
        int n = 0;
        if (cudaOccupancyMaxActiveClusters(&n, attn_block_tc_kernel, &cfg) == cudaSuccess && n > 0) max_clusters_dev[dev] = n;
        else { max_clusters_dev[dev] = 0; cudaGetLastError(); }
        done_dev[dev] = true;
      }
    }
  }
  const int max_clusters = max_clusters_dev[dev];
  TCS_CUDA(attr_err);
  int ncl = sm_count / 2;
  if (max_clusters > 0 && max_clusters < ncl) ncl = max_clusters;
  if (ncl > p.B) ncl = p.B;
  if (ncl < 1) ncl = 1;
  typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                      const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                      CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static PFN_encodeTiled encode = nullptr;
  if (!encode) {
    void* fp = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fp, cudaEnableDefault, &q) != cudaSuccess || !fp)
      return fail(TCS_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
    encode = reinterpret_cast<PFN_encodeTiled>(fp);
  }
  AttnTcMaps maps;
  {
    const cuuint64_t dims[4] = {192, 18, 18, static_cast<cuuint64_t>(p.B)};
    const cuuint64_t strides[3] = {384, 18 * 384, 18 * 18 * 384};
    const cuuint32_t es[4] = {1, 1, 1, 1};
    const cuuint32_t box8[4] = {64, 16, 8, 1}, box1[4] = {64, 16, 1, 1};
    auto mk = [&](CUtensorMap* m, const void* base, const cuuint32_t* box) {
      return encode(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, es,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    };
    if (mk(&maps.x, p.x, box8) != CUDA_SUCCESS || mk(&maps.out, p.out, box8) != CUDA_SUCCESS ||
        mk(&maps.out_row, p.out, box1) != CUDA_SUCCESS)
      return fail(TCS_ERR_CUDA, "attn_tc: cuTensorMapEncodeTiled failed");
  }
  attn_block_tc_kernel<<<2 * ncl, AT_THREADS, smem, st>>>(maps, p);
  TCS_CUDA(cudaGetLastError());
  return TCS_OK;
}

}  // namespace tcs
