// linear_tc.cu — nn.Linear as a tcgen05 GEMM for the latent diffusion prior (SURVEY 8f-1).
//
// Replaces the F.linear calls of DiffusionPriorFiLM / FiLMResBlock (reference:
// src/toycrystals/models/diffusion_prior.py:43-54 fc1/fc2/cond, :86-97 y_fuse/t_mlp) for bf16 operands:
//
//   out[M, N] = act(A[M, K] · W[N, K]^T + bias[N])
//
// * A (activations) and W (the nn.Linear weight, already [out, in] = K-major) are bf16; TMA (SWIZZLE_128B, 64-element
//   = 128-byte K slabs) stages 128 x 64 A tiles and 256 x 64 W tiles in a 4-6 deep mbarrier ring;
// * one elected thread issues tcgen05.mma kind::f16 (M = 128 per CTA, N = 256, K = 16), fp32 accumulators in TMEM,
//   two 256-column sets so the epilogue of tile i overlaps the main loop of tile i+1;
// * CTA pairs (cluster of 2, cta_group::2): the pair shares the N tile, each CTA loads only half of the W tile
//   (128 rows) and the leader's MMA (M = 256) reads it half from each CTA's shared memory;
// * epilogue warps (4) read TMEM with tcgen05.ld, apply bias / SiLU, stage 32 x 32 blocks in swizzled shared-memory
//   slabs and hand them to the TMA unit: a tensor store for fc1 (bf16) and a tensor REDUCE-ADD for fc2, so the fp32
//   residual stream h += ... is accumulated at L2 without the kernel ever reading h (one row per lane straight to
//   global memory cost 32 cache-line requests per instruction and made the epilogue, not the MMA, the bottleneck);
// * persistent grid, one CTA per SM.
//
// CONV = true turns the same kernel into ConvTranspose2d(k = 4, s = 2, p = 1) + ReLU of the CondVAE decoder
// (src/toycrystals/models/vae.py:36-43): each of the 4 output parity classes (oy & 1, ox & 1) is a 2x2-tap stride-1
// convolution, i.e. a GEMM with K = 4 taps x C_in whose A rows are the input pixels shifted by the tap offset.  The
// activations are NHWC bf16 and TMA fetches a tap as a 4-D box (channels, x, y, image) at shifted coordinates; the
// zero fill TMA applies outside the tensor IS the transposed convolution's implicit zero border.
#include "linear_tc.cuh"

#include "tc_ptx.cuh"

namespace tcs {

constexpr int LT_BM = 128, LT_BN = 256, LT_BK = 64;
constexpr int LT_EPI_WARPS = 8;
constexpr int LT_THREADS = 64 + 32 * LT_EPI_WARPS;   // TMA warp, MMA warp, 8 epilogue warps (2 per TMEM lane quarter)
constexpr int LT_MAX_STAGES = 8;
constexpr uint32_t LT_SLAB_BYTES = LT_EPI_WARPS * 8192;   // TMA-store staging: 2 x 4 KB per epilogue warp
constexpr uint32_t LT_BIAS_BYTES = 2 * 256 * 4;            // bias of the current N tile, one copy per accumulator set

struct __align__(8) LtBarriers {
  uint64_t full[LT_MAX_STAGES];
  uint64_t empty[LT_MAX_STAGES];
  uint64_t tmem_full[2];
  uint64_t tmem_empty[2];
  uint32_t tmem_base;
};

__device__ __forceinline__ float lt_silu(float y) {   // y * sigmoid(y) = h + h tanh(h), h = y / 2 (one MUFU)
  const float h = 0.5f * y;
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
  return fmaf(h, t, h);
}
__device__ __forceinline__ uint32_t lt_pack(float a, float b) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&h);
}

// tile -> (M tile, N tile [for CONV: N tile index = parity class, the weight matrices of the 4 classes are stacked]);
// the two CTAs of a pair (consecutive tile indices) share the N tile
__device__ __forceinline__ void lt_tile_to_mn(int tile, int n_mtiles, int& mt, int& nt) {
  const int pt = tile >> 1, half = n_mtiles >> 1;
  nt = pt / half;
  mt = ((pt - nt * half) << 1) | (tile & 1);
}
// transposed-conv tap (ty, tx) of parity (py, px): input offset per axis
__device__ __forceinline__ int lt_tap_off(int parity_bit, int tap_bit) {
  return parity_bit == 0 ? (tap_bit == 0 ? 0 : -1) : (tap_bit == 0 ? 1 : 0);
}

template <int BN, bool CONV>
__global__ void __launch_bounds__(LT_THREADS, 1)
linear_tc_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapW,
                 const __grid_constant__ CUtensorMap mapO, const LinearTcParams p) {
  constexpr int LT_BN = BN;          // N tile of this instance (accumulator sets stay 256 TMEM columns apart)
  constexpr int ACC_COLS = 256;
  extern __shared__ uint8_t smem_raw[];
  __shared__ LtBarriers bars;
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;   // warp-uniform for the compiler
  const uint32_t smem_base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  const int n_tiles = p.n_mtiles * p.n_ntiles;
  constexpr int NB = LT_BN / 2;                  // W rows this CTA stages per K block
  constexpr uint32_t B_BYTES = NB * LT_BK * 2;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&mapA);
    ptx::prefetch_tmap(&mapW);
    if (!CONV) ptx::prefetch_tmap(&mapO);
    for (int s = 0; s < p.nstage; ++s) {
      ptx::mbar_init(ptx::smem_u32(&bars.full[s]), 1);
      ptx::mbar_init(ptx::smem_u32(&bars.empty[s]), 1);
    }
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(ptx::smem_u32(&bars.tmem_full[a]), 1);
      ptx::mbar_init(ptx::smem_u32(&bars.tmem_empty[a]), LT_EPI_WARPS * 2);
    }
    ptx::fence_barrier_init();
  }
  const uint32_t cta_rank = ptx::cluster_ctarank();
  if (warp == 1) ptx::tmem_alloc_512_2sm(ptx::smem_u32(&bars.tmem_base));
  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync_all();
  ptx::tc_fence_after();
  const uint32_t tmem_base = bars.tmem_base;

  if (warp == 0) {
    // ============================== TMA producer ==============================
    uint32_t stage = 0, phase = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      int mt, nt;
      lt_tile_to_mn(tile, p.n_mtiles, mt, nt);
      // CONV: the 128 rows of an M tile are `imgs` whole images (Hi*Hi < 128) or `rows_y` rows of one image
      int b0 = 0, y0 = 0;
      if (CONV) {
        if (p.tiles_per_img > 1) { b0 = mt / p.tiles_per_img; y0 = (mt - b0 * p.tiles_per_img) * p.rows_y; }
        else b0 = mt * p.imgs;
      }
      for (int kb = 0; kb < p.kblocks; ++kb) {
        ptx::mbar_wait(ptx::smem_u32(&bars.empty[stage]), phase ^ 1);
        if (lane == 0) {
          const uint32_t full = ptx::smem_u32(&bars.full[stage]);
          const uint32_t a_dst = smem_base + stage * p.stage_bytes;
          const uint32_t b_dst = a_dst + p.a_bytes;
          if (cta_rank == 0) ptx::mbar_expect_tx(full, 2 * (p.a_bytes + B_BYTES));
          if (CONV) {
            const int tap = kb / p.cblocks, cb = kb - tap * p.cblocks;
            const int dy = lt_tap_off(nt >> 1, tap >> 1), dx = lt_tap_off(nt & 1, tap & 1);
            ptx::tma_load_4d_2sm(a_dst, &mapA, full, cb * LT_BK, dx, y0 + dy, b0);
          } else {
            ptx::tma_load_2d_2sm(a_dst, &mapA, full, kb * LT_BK, mt * LT_BM);
          }
          ptx::tma_load_2d_2sm(b_dst, &mapW, full, kb * LT_BK, nt * LT_BN + static_cast<int>(cta_rank) * NB);
        }
        __syncwarp();
        if (++stage == static_cast<uint32_t>(p.nstage)) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1 && cta_rank == 0) {
    // ============================== MMA issuer (leader CTA only) =================
    constexpr uint32_t idesc = make_idesc(LT_BM * 2, LT_BN);
    uint32_t stage = 0, phase = 0, acc = 0, acc_phase = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      ptx::mbar_wait(ptx::smem_u32(&bars.tmem_empty[acc]), acc_phase ^ 1);
      ptx::tc_fence_after();
      const uint32_t d_tmem = tmem_base + acc * ACC_COLS;
      for (int kb = 0; kb < p.kblocks; ++kb) {
        ptx::mbar_wait(ptx::smem_u32(&bars.full[stage]), phase);
        ptx::tc_fence_after();
        if (lane == 0) {
          const uint32_t a_base = smem_base + stage * p.stage_bytes;
          const uint64_t adesc = make_desc_sw128(a_base), bdesc = make_desc_sw128(a_base + p.a_bytes);
#pragma unroll
          for (int k = 0; k < LT_BK / 16; ++k) {   // 32 bytes per K = 16 step inside the 128-byte swizzle row
            const uint32_t accum = (kb | k) != 0 ? 1u : 0u;
            ptx::umma_bf16_2sm(d_tmem, adesc + k * 2, bdesc + k * 2, idesc, accum);
          }
          ptx::umma_commit_2sm(ptx::smem_u32(&bars.empty[stage]));
          if (kb == p.kblocks - 1) ptx::umma_commit_2sm(ptx::smem_u32(&bars.tmem_full[acc]));
        }
        __syncwarp();
        if (++stage == static_cast<uint32_t>(p.nstage)) { stage = 0; phase ^= 1; }
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
  } else if (warp >= 2) {
    // ============================== epilogue: warp reads TMEM lane quarter q = warp % 4, column half (warp-2)/4 ====
    const int q = warp & 3, half = (warp - 2) >> 2;
    constexpr int NC = LT_BN / 32;                       // 32-column chunks per tile
    constexpr int CPW = NC >= 2 ? NC / 2 : 1;            // chunks per warp
    const int c_begin = NC >= 2 ? half * CPW : 0;
    const bool has_work = NC >= 2 || half == 0;
    uint32_t acc = 0, acc_phase = 0, slab_buf = 0;
    // TMA-store staging: 2 x 4 KB per epilogue warp after the operand ring (1024-byte aligned), then the bias
    const uint32_t slab = smem_base + p.nstage * p.stage_bytes + static_cast<uint32_t>(warp - 2) * 8192;
    float* bias_s = reinterpret_cast<float*>(smem_raw + (smem_base - ptx::smem_u32(smem_raw)) + p.nstage * p.stage_bytes + LT_SLAB_BYTES);
    const int et = threadIdx.x - 64;                     // 0..255 among the epilogue threads
    (void)slab; (void)slab_buf;
    const bool silu = (p.flags & LIN_SILU) != 0, f32 = (p.flags & LIN_OUT_F32) != 0, accum = (p.flags & LIN_ACCUM) != 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      int mt, nt;
      lt_tile_to_mn(tile, p.n_mtiles, mt, nt);
      const int r = q * 32 + lane;
      size_t row = static_cast<size_t>(mt) * LT_BM + r;     // output row (pixel) index
      bool live = row < static_cast<size_t>(p.M);
      if (CONV) {   // input pixel (b, i, j) -> output pixel (2i + py, 2j + px)
        int b, i, j;
        const int Hi = p.Hi;
        if (p.tiles_per_img > 1) {
          b = mt / p.tiles_per_img;
          i = (mt - b * p.tiles_per_img) * p.rows_y + r / Hi;
          j = r % Hi;
        } else {
          const int bi = r / (Hi * Hi), rem = r - bi * Hi * Hi;
          b = mt * p.imgs + bi; i = rem / Hi; j = rem - i * Hi;
        }
        live = b < p.n_img;
        row = (static_cast<size_t>(b) * 2 * Hi + 2 * i + (nt >> 1)) * 2 * Hi + 2 * j + (nt & 1);
      }
      const int col0 = CONV ? 0 : nt * LT_BN;
      const bool relu = (p.flags & LIN_RELU_TC) != 0;
      const uint32_t tbase = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * ACC_COLS;
      // bias of this N tile -> shared memory (while the main loop of the tile is still running)
      float* bs = bias_s + acc * 256;
      if (et < LT_BN) bs[et] = p.bias ? __ldg(p.bias + col0 + et) : 0.f;
      asm volatile("bar.sync 1, %0;" ::"n"(32 * LT_EPI_WARPS) : "memory");
      ptx::mbar_wait(ptx::smem_u32(&bars.tmem_full[acc]), acc_phase);
      ptx::tc_fence_after();
      float vbuf[2][32];
      if (has_work) ptx::tmem_ld32(tbase + c_begin * 32, vbuf[0]);
#pragma unroll
      for (int cc = 0; cc < CPW; ++cc) {
        if (!has_work) break;
        const int c = c_begin + cc;
        ptx::tmem_ld_wait();
        if (cc + 1 < CPW) ptx::tmem_ld32(tbase + (c + 1) * 32, vbuf[(cc + 1) & 1]);
        float* v = vbuf[cc & 1];
        const int col = col0 + c * 32;
        {
#pragma unroll
          for (int i = 0; i < 32; i += 4) {
            const float4 b4 = *reinterpret_cast<const float4*>(bs + c * 32 + i);
            v[i] += b4.x; v[i + 1] += b4.y; v[i + 2] += b4.z; v[i + 3] += b4.w;
          }
        }
        if (silu) {
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = lt_silu(v[i]);
        }
        if (relu) {
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i], 0.f);
        }
        if (!CONV) {
          // 32 rows x 32 columns -> swizzled slab -> one TMA store / reduce-add per block (full 128-byte lines)
          if (lane == 0) ptx::bulk_wait_read<1>();   // the slab half written two blocks ago has been read
          __syncwarp();
          const uint32_t base = slab + slab_buf * 4096;
          if (f32) {
            const uint32_t dst = base + lane * 128;
#pragma unroll
            for (int j = 0; j < 8; ++j)
              ptx::st_shared_v4(dst + ((j ^ (lane & 7)) << 4), v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
          } else {
            const uint32_t dst = base + lane * 64;
            const int sw = (lane >> 1) & 3;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const uint32_t a0 = lt_pack(v[8 * j], v[8 * j + 1]), a1 = lt_pack(v[8 * j + 2], v[8 * j + 3]);
              const uint32_t a2 = lt_pack(v[8 * j + 4], v[8 * j + 5]), a3 = lt_pack(v[8 * j + 6], v[8 * j + 7]);
              asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst + ((j ^ sw) << 4)), "r"(a0), "r"(a1), "r"(a2), "r"(a3) : "memory");
            }
          }
          ptx::fence_proxy_async();
          __syncwarp();
          if (lane == 0) {
            const int r0 = mt * LT_BM + q * 32;
            if (r0 < p.M) {   // rows past M inside the box are clipped by the tensor map
              if (accum) ptx::tma_reduce_add_2d(&mapO, base, col, r0);
              else ptx::tma_store_2d(&mapO, base, col, r0);
            }
            ptx::bulk_commit();
          }
          slab_buf ^= 1;
        } else if (live && f32) {
          float* o = static_cast<float*>(p.out) + row * p.ldo + col;
#pragma unroll
          for (int i = 0; i < 32; i += 4) {
            float4 r = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
            if (accum) {
              const float4 a4 = *reinterpret_cast<const float4*>(o + i);
              r.x += a4.x; r.y += a4.y; r.z += a4.z; r.w += a4.w;
            }
            *reinterpret_cast<float4*>(o + i) = r;
          }
        } else if (live) {
          uint4* o = reinterpret_cast<uint4*>(static_cast<__nv_bfloat16*>(p.out) + row * p.ldo + col);
#pragma unroll
          for (int i = 0; i < 32; i += 8)
            o[i / 8] = make_uint4(lt_pack(v[i], v[i + 1]), lt_pack(v[i + 2], v[i + 3]), lt_pack(v[i + 4], v[i + 5]),
                                  lt_pack(v[i + 6], v[i + 7]));
        }
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive_rank0(ptx::smem_u32(&bars.tmem_empty[acc]));
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
    if (!CONV && lane == 0) ptx::bulk_wait_all();   // staged TMA stores have completed
  }

  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync_all();   // the leader's MMAs read the peer's shared memory / write its TMEM
  ptx::tc_fence_after();
  if (warp == 1) ptx::tmem_dealloc_512_2sm(tmem_base);
}

// ---------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static PFN_encodeTiled lt_get_encode() {
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

static int lt_encode_2d(CUtensorMap* map, const __nv_bfloat16* base, int rows, int cols, int pitch, int box_rows) {
  PFN_encodeTiled encode = lt_get_encode();
  if (!encode) return fail(TCS_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(pitch) * 2};
  cuuint32_t box[2] = {LT_BK, static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<__nv_bfloat16*>(base), dims, strides, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(TCS_ERR_CUDA, "cuTensorMapEncodeTiled(linear) failed: " + std::to_string(r));
  return TCS_OK;
}

int linear_tc_make_plan(LinearTcPlan* plan, const __nv_bfloat16* A, int lda, const __nv_bfloat16* W, int ldw, int M, int N,
                        int K, const float* bias, void* out, int ldo, int flags, int sm_count) {
  if (M < 1 || N % LT_BN || K % LT_BK || K < LT_BK)
    return fail(TCS_ERR_UNSUPPORTED, "linear_tc: needs N % 256 == 0 and K % 64 == 0 (got N=" + std::to_string(N) +
                                         ", K=" + std::to_string(K) + ")");
  if ((lda % 8) || (ldw % 8) || (reinterpret_cast<uintptr_t>(A) & 15) || (reinterpret_cast<uintptr_t>(W) & 15))
    return fail(TCS_ERR_BAD_ARGUMENT, "linear_tc: operands must be 16-byte aligned with 16-byte row pitches");
  if ((flags & LIN_ACCUM) && !(flags & LIN_OUT_F32)) return fail(TCS_ERR_BAD_ARGUMENT, "linear_tc: accumulate needs fp32 output");
  LinearTcPlan& pl = *plan;
  pl = LinearTcPlan();
  pl.bn = LT_BN;
  pl.conv = false;
  LinearTcParams& p = pl.p;
  p = LinearTcParams();
  p.M = M; p.N = N; p.K = K;
  p.n_mtiles = (M + LT_BM - 1) / LT_BM;
  if (p.n_mtiles & 1) ++p.n_mtiles;   // whole CTA pairs: the extra tile is all out-of-bounds rows
  p.n_ntiles = N / LT_BN;
  p.kblocks = K / LT_BK;
  p.a_bytes = LT_BM * LT_BK * 2;
  p.stage_bytes = p.a_bytes + (LT_BN / 2) * LT_BK * 2;
  const size_t budget = 227 * 1024 - 2048 - 1024 - LT_SLAB_BYTES - LT_BIAS_BYTES;
  p.nstage = static_cast<int>(budget / p.stage_bytes);
  if (p.nstage > LT_MAX_STAGES) p.nstage = LT_MAX_STAGES;
  pl.smem = static_cast<size_t>(p.nstage) * p.stage_bytes + 1024 + LT_SLAB_BYTES + LT_BIAS_BYTES;
  p.bias = bias; p.out = out; p.ldo = ldo; p.flags = flags;
  const int tiles = p.n_mtiles * p.n_ntiles;
  pl.grid = (tiles < sm_count ? tiles : sm_count) & ~1;
  TCS_CHECK(lt_encode_2d(&pl.mapA, A, M, K, lda, LT_BM));
  TCS_CHECK(lt_encode_2d(&pl.mapW, W, N, K, ldw, LT_BN / 2));
  {   // output: 32-column x 32-row boxes, written (bf16 / fp32) or reduce-added (fp32) by TMA from swizzled slabs
    PFN_encodeTiled encode = lt_get_encode();
    const bool f32 = (flags & LIN_OUT_F32) != 0;
    if ((reinterpret_cast<uintptr_t>(out) & 15) || (static_cast<size_t>(ldo) * (f32 ? 4 : 2)) % 16)
      return fail(TCS_ERR_BAD_ARGUMENT, "linear_tc: the output must be 16-byte aligned with a 16-byte row pitch");
    cuuint64_t dims[2] = {static_cast<cuuint64_t>(N), static_cast<cuuint64_t>(M)};
    cuuint64_t strides[1] = {static_cast<cuuint64_t>(ldo) * (f32 ? 4 : 2)};
    cuuint32_t box[2] = {32, 32};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = encode(&pl.mapO, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, out, dims, strides,
                        box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, f32 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(TCS_ERR_CUDA, "cuTensorMapEncodeTiled(linear out) failed: " + std::to_string(r));
  }
  pl.valid = true;
  return TCS_OK;
}

static int lt_encode_4d(CUtensorMap* map, const __nv_bfloat16* base, int n, int Hi, int Ci, int box_y, int box_b) {
  PFN_encodeTiled encode = lt_get_encode();
  if (!encode) return fail(TCS_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  const cuuint64_t C = static_cast<cuuint64_t>(Ci);
  cuuint64_t dims[4] = {C, static_cast<cuuint64_t>(Hi), static_cast<cuuint64_t>(Hi), static_cast<cuuint64_t>(n)};
  cuuint64_t strides[3] = {C * 2, C * 2 * Hi, C * 2 * Hi * Hi};
  cuuint32_t box[4] = {LT_BK, static_cast<cuuint32_t>(Hi), static_cast<cuuint32_t>(box_y), static_cast<cuuint32_t>(box_b)};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<__nv_bfloat16*>(base), dims, strides, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(TCS_ERR_CUDA, "cuTensorMapEncodeTiled(convT input) failed: " + std::to_string(r));
  return TCS_OK;
}

int linear_tc_make_convt_plan(LinearTcPlan* plan, const __nv_bfloat16* in, const __nv_bfloat16* wpacked, const float* bias,
                              int n, int Hi, int Ci, int Co, __nv_bfloat16* out, int sm_count) {
  if (n < 1 || (Hi != 4 && Hi != 8 && Hi != 16) || Ci % LT_BK || (Co != 32 && Co != 64 && Co != 128))
    return fail(TCS_ERR_UNSUPPORTED, "linear_tc convT: needs Hi in {4,8,16}, C_in % 64 == 0, C_out in {32,64,128}");
  LinearTcPlan& pl = *plan;
  pl = LinearTcPlan();
  pl.bn = Co;
  pl.conv = true;
  LinearTcParams& p = pl.p;
  p = LinearTcParams();
  p.Hi = Hi; p.n_img = n; p.cblocks = Ci / LT_BK;
  const int pix = Hi * Hi;
  if (pix >= LT_BM) { p.tiles_per_img = pix / LT_BM; p.rows_y = LT_BM / Hi; p.imgs = 1; }
  else { p.tiles_per_img = 1; p.rows_y = Hi; p.imgs = LT_BM / pix; }
  p.n_mtiles = pix >= LT_BM ? n * p.tiles_per_img : (n + p.imgs - 1) / p.imgs;
  if (p.n_mtiles & 1) ++p.n_mtiles;
  p.M = p.n_mtiles * LT_BM;           // liveness is decided per image in the epilogue
  p.N = Co; p.K = 4 * Ci;
  p.n_ntiles = 4;                     // the parity classes
  p.kblocks = 4 * p.cblocks;
  p.a_bytes = LT_BM * LT_BK * 2;
  p.stage_bytes = p.a_bytes + (Co / 2) * LT_BK * 2;
  const size_t budget = 227 * 1024 - 2048 - 1024 - LT_SLAB_BYTES - LT_BIAS_BYTES;
  p.nstage = static_cast<int>(budget / p.stage_bytes);
  if (p.nstage > LT_MAX_STAGES) p.nstage = LT_MAX_STAGES;
  pl.smem = static_cast<size_t>(p.nstage) * p.stage_bytes + 1024 + LT_SLAB_BYTES + LT_BIAS_BYTES;
  p.bias = bias; p.out = out; p.ldo = Co; p.flags = LIN_RELU_TC;
  const int tiles = p.n_mtiles * p.n_ntiles;
  pl.grid = (tiles < sm_count ? tiles : sm_count) & ~1;
  TCS_CHECK(lt_encode_4d(&pl.mapA, in, n, Hi, Ci, p.rows_y, p.imgs));
  TCS_CHECK(lt_encode_2d(&pl.mapW, wpacked, 4 * Co, 4 * Ci, 4 * Ci, Co / 2));
  pl.mapO = pl.mapW;   // unused: the scattered (stride-2 pixel) rows are stored per lane
  pl.valid = true;
  return TCS_OK;
}

template <int BN, bool CONV>
static int lt_launch_t(const LinearTcPlan& pl, cudaStream_t st) {
  auto kern = linear_tc_kernel<BN, CONV>;
  static bool attr_done = false;
  if (!attr_done) {
    TCS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024 - 2048));
    attr_done = true;
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(pl.grid); cfg.blockDim = dim3(LT_THREADS); cfg.dynamicSmemBytes = pl.smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  TCS_CUDA(cudaLaunchKernelEx(&cfg, kern, pl.mapA, pl.mapW, pl.mapO, pl.p));
  TCS_CUDA(cudaGetLastError());
  return TCS_OK;
}

int linear_tc_launch(const LinearTcPlan& pl, cudaStream_t st) {
  if (!pl.valid) return fail(TCS_ERR_STATE, "linear_tc_launch: plan not built");
  if (pl.conv) {
    if (pl.bn == 128) return lt_launch_t<128, true>(pl, st);
    if (pl.bn == 64) return lt_launch_t<64, true>(pl, st);
    return lt_launch_t<32, true>(pl, st);
  }
  return lt_launch_t<256, false>(pl, st);
}

}  // namespace tcs
