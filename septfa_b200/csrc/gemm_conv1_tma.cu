// TMA-fed persistent tcgen05 kernel for the first contraction of a TCN block (model/model.py:132/138) in the
// half-stream mode of the forward (blocks 1 .. n-1: the residual stream travels as fp16 [M,256], written by the
// cluster-resident residual kernel):
//   p = PReLU(W1 GN(stream) + b1),  statistics of p
// The GroupNorm of the stream is taken OUT of the A operand: with W' = W1 diag(gamma) (folded at load time) and the raw
// stream w,   W' ((w - mean) rstd) + b' = rstd (W' w) + (b' - rstd mean S),   S[n] = sum_k W'[n,k]  (of the fp16 image),
// so the A operand is the stored stream itself and no thread touches it on its way to the tensor core: one TMA tensor
// load (2-D box 64 halves x 128 rows, 128-byte swizzle) per K-chunk lands in shared memory already in the K-major
// SWIZZLE_128B operand layout. The whole weight image (128 KB) is loaded once per CTA and stays resident, so the only
// per-tile traffic into the SM is the tile's 64 KB of stream. Roles (one CTA per SM, 12 warps):
//   warp 0       TMA producer : ring of 5 A stages (16 KB each), runs ahead across tile boundaries
//   warp 1       MMA issuer   : tcgen05.mma 128x256x16, double-buffered TMEM accumulator (2 x 256 columns)
//   warps 4-11   epilogue     : tcgen05.ld -> rstd * acc + (b' - rstd mean S) -> PReLU -> statistics -> fp16 -> K-group planes
//                               of p (kernels.h, DconvMmaParams); a lane = a row, 32 lanes = 512 contiguous bytes per plane
// Synchronisation is mbarriers only. Requires T >= 128 (a tile touches at most two utterances).
#include <algorithm>
#include <cuda.h>
#include "kernels.h"
#include "tc_common.cuh"

namespace septfa {

namespace {

using namespace tc;

constexpr int kTileM = 128;
constexpr int kNCH = 4;                       // K = 256 = 4 chunks of 64
constexpr int kAStages = 5;
constexpr int kABytes = kTileM * 128;         // 16 KB: 128 rows x 64 halves
constexpr int kWBytes = 256 * 128;            // 32 KB: 256 rows x 64 halves
constexpr int kOffA = 0;
constexpr int kOffW = kOffA + kAStages * kABytes;            // 80 KB
constexpr int kOffSb = kOffW + kNCH * kWBytes;               // + 128 KB
constexpr int kOffBar = kOffSb + 2048;
constexpr int kSmemBytes = kOffBar + 256;
constexpr int kEpiWarps = 8;                  // 4 TMEM lane quarters x 2 column halves
constexpr int kEpiCols = 256 / (kEpiWarps / 4);
constexpr int kThreadsT = (4 + kEpiWarps) * 32;
static_assert(kOffW % 1024 == 0 && kSmemBytes <= 232448, "shared-memory plan");

struct TmaParams {
  alignas(64) CUtensorMap a_tmap;   // the stream: fp16 [M rows][256], box 64 x 128, SWIZZLE_128B
  int M, T, ntiles, Mp;
  const __half* w_img;              // 4 K-chunks x [256 rows x 128 B], 128B-swizzled K-major
  const float4* sb;                 // [128] {S[2i], S[2i+1], b'[2i], b'[2i+1]}
  const Stat2* st_in;               // [B] statistics of the stream (nullptr: no norm, y = w)
  double inv_n; float eps;
  float slope;
  __half* out;                      // K-group planes [32][Mp][8]
  Stat2* st_out;                    // [B]
};

__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* tmap, int c0, int c1, uint64_t* bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
                   smem_u32(dst)),
               "l"(tmap), "r"(c0), "r"(c1), "r"(smem_u32(bar))
               : "memory");
}

template <bool AMAX>
__global__ void __launch_bounds__(kThreadsT, 1) k_conv1_tma(const __grid_constant__ TmaParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kOffBar);
  uint64_t* a_full = bars;                    // [5] TMA bytes
  uint64_t* a_empty = bars + 5;               // [5] MMA commit
  uint64_t* w_full = bars + 10;               // [4] bulk copy bytes (once)
  uint64_t* acc_full = bars + 14;             // [2] MMA commit
  uint64_t* acc_empty = bars + 16;            // [2] kEpiWarps * 32 epilogue arrivals
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 18);
  const float4* sb_s = reinterpret_cast<const float4*>(smem + kOffSb);
  constexpr uint32_t IDESC = make_idesc_f16(kTileM, 256);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    if ((smem_u32(smem) & 1023u) != 0u) __trap();
    for (int s = 0; s < kAStages; ++s) { mbar_init(a_full + s, 1); mbar_init(a_empty + s, 1); }
    for (int j = 0; j < kNCH; ++j) mbar_init(w_full + j, 1);
    for (int s = 0; s < 2; ++s) { mbar_init(acc_full + s, 1); mbar_init(acc_empty + s, kEpiWarps * 32); }
    fence_mbar_init();
    // static weights: the whole image, once, before the dependency wait
    for (int j = 0; j < kNCH; ++j) {
      mbar_expect_tx(w_full + j, kWBytes);
      bulk_copy_g2s(smem + kOffW + j * kWBytes, reinterpret_cast<const uint8_t*>(p.w_img) + (size_t)j * kWBytes, kWBytes, w_full + j);
    }
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  if (threadIdx.x < 128) reinterpret_cast<float4*>(smem + kOffSb)[threadIdx.x] = __ldg(p.sb + threadIdx.x);
  pdl_launch_dependents();
  pdl_wait();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int first = blockIdx.x, stride = gridDim.x;

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer (rows past M read as zeros)
    if (lane == 0) {
      int g = 0;
      for (int tile = first; tile < p.ntiles; tile += stride) {
        for (int j = 0; j < kNCH; ++j, ++g) {
          const int s = g % kAStages, u = g / kAStages;
          if (u > 0) mbar_wait(a_empty + s, (u - 1) & 1, 100 + j);
          mbar_expect_tx(a_full + s, kABytes);
          tma_load_2d(smem + kOffA + s * kABytes, &p.a_tmap, j * 64, tile * kTileM, a_full + s);
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer
    if (lane == 0) {
      int g = 0, lt = 0;
      for (int tile = first; tile < p.ntiles; tile += stride, ++lt) {
        const int buf = lt & 1, ub = lt >> 1;
        if (ub > 0) { mbar_wait(acc_empty + buf, (ub - 1) & 1, 600); tc_fence_after(); }
        for (int j = 0; j < kNCH; ++j, ++g) {
          const int sa = g % kAStages, ua = g / kAStages;
          if (lt == 0) mbar_wait(w_full + j, 0, 200 + j);
          mbar_wait(a_full + sa, ua & 1, 300 + j);
          tc_fence_after();
          const uint64_t a_desc = make_sw128_desc(smem_u32(smem + kOffA + sa * kABytes));
          const uint64_t b_desc = make_sw128_desc(smem_u32(smem + kOffW + j * kWBytes));
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)
            umma_f16(tmem_base + (uint32_t)(buf * 256), a_desc + (uint64_t)(kk * 2), b_desc + (uint64_t)(kk * 2), IDESC, (j | kk) != 0);
          umma_commit(a_empty + sa);
        }
        umma_commit(acc_full + buf);
      }
    }
    __syncwarp();
  } else if (warp >= 4) {
    // ------------------------------------------------------------ epilogue: kEpiWarps = 4 lane quarters x column parts
    const int lq = warp & 3, ch = (warp - 4) >> 2;
    const int rl = lq * 32 + lane;                           // a lane = a row of the tile
    const float2 sl2 = make_float2(p.slope, p.slope);
    const bool has_norm = p.st_in != nullptr;
    // mean / rstd of a tile's (at most two) utterances: lanes 0 / 1 compute (double arithmetic behind two L2 loads), the
    // warp reads them by shuffle. Computed one tile AHEAD, under the tensor-memory loads of the current tile.
    auto tile_stats = [&](int tile) -> float2 {
      float2 mr = make_float2(0.f, 1.f);
      if (tile < p.ntiles && has_norm && lane < 2) {
        const int r0 = tile * kTileM, nrows = min(kTileM, p.M - r0);
        const int b_first = r0 / p.T, e1 = (b_first + 1) * p.T;
        if (lane == 0 || e1 < r0 + nrows) mr = stat_mean_rstd(p.st_in + b_first + lane, p.inv_n, p.eps);
      }
      return mr;
    };
    float2 mr = tile_stats(first);
    int lt = 0;
    for (int tile = first; tile < p.ntiles; tile += stride, ++lt) {
      const int buf = lt & 1;
      const int r0 = tile * kTileM, nrows = min(kTileM, p.M - r0);
      const int b_first = r0 / p.T, e1 = (b_first + 1) * p.T;   // first row of the tile's second utterance
      const float m0 = __shfl_sync(0xffffffffu, mr.x, 0), s0 = __shfl_sync(0xffffffffu, mr.y, 0);
      const float m1 = __shfl_sync(0xffffffffu, mr.x, 1), s1 = __shfl_sync(0xffffffffu, mr.y, 1);
      const bool valid = rl < nrows, second = r0 + rl >= e1;
      const float mean = second ? m1 : m0, rstd = second ? s1 : s0;
      const float2 rs2 = make_float2(rstd, rstd), nr2 = make_float2(-mean * rstd, -mean * rstd);
      mbar_wait(acc_full + buf, (lt >> 1) & 1, 500);
      tc_fence_after();
      float2 s2 = make_float2(0.f, 0.f), q2 = make_float2(0.f, 0.f);
      const uint32_t t_row = tmem_base + (uint32_t)(buf * 256) + ((uint32_t)(lq * 32) << 16) + (uint32_t)(ch * kEpiCols);
      auto process = [&](const uint32_t (&u)[32], int c) {
        const int cc = ch * (kEpiCols / 32) + c, col0 = cc * 32;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          uint32_t h[4];
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const float4 t4 = sb_s[(col0 >> 1) + i * 4 + k];   // same address in every lane: broadcast
            const float2 k0 = __ffma2_rn(nr2, make_float2(t4.x, t4.y), make_float2(t4.z, t4.w));
            const float2 x = __ffma2_rn(rs2, make_float2(__uint_as_float(u[8 * i + 2 * k]), __uint_as_float(u[8 * i + 2 * k + 1])), k0);
            const float2 ax = __fmul2_rn(sl2, x);
            float2 y;
            if constexpr (AMAX) y = make_float2(fmaxf(x.x, ax.x), fmaxf(x.y, ax.y));
            else y = make_float2(fminf(x.x, ax.x), fminf(x.y, ax.y));
            s2 = __fadd2_rn(s2, y);
            q2 = __ffma2_rn(y, y, q2);
            h[k] = pack_half2(y.x, y.y);
          }
          if (valid)
            *reinterpret_cast<uint4*>(p.out + ((size_t)(cc * 4 + i) * p.Mp + (size_t)(kPlaneHalo + r0 + rl)) * 8) =
                make_uint4(h[0], h[1], h[2], h[3]);
        }
      };
      // two tensor-memory loads in flight (the next 32 columns arrive while the current ones are finished); the next tile's
      // statistics are computed under the first pair
      constexpr int NC = kEpiCols / 32;
      uint32_t va[32], vb[32];
      tmem_ld32_nowait(t_row, va);
      tmem_ld32_nowait(t_row + 32u, vb);
      mr = tile_stats(tile + stride);
#pragma unroll
      for (int c2 = 0; c2 < NC / 2; ++c2) {
        tmem_ld_wait();                // va and vb (chunks 2 c2, 2 c2 + 1) have landed
        if (c2 + 1 == NC / 2) {        // this warp's part of the accumulator is in registers
          tc_fence_before();
          mbar_arrive(acc_empty + buf);
        }
        process(va, 2 * c2);
        if (c2 + 1 < NC / 2) tmem_ld32_nowait(t_row + (uint32_t)((2 * c2 + 2) * 32), va);
        process(vb, 2 * c2 + 1);
        if (c2 + 1 < NC / 2) tmem_ld32_nowait(t_row + (uint32_t)((2 * c2 + 3) * 32), vb);
      }
      // statistics of this warp's 32 rows x kEpiCols columns, per utterance: fixed-order shuffle trees, one double atomic pair
      const float sv = valid ? s2.x + s2.y : 0.f, qv = valid ? q2.x + q2.y : 0.f;
      const float a0 = warp_sum(second ? 0.f : sv), c0 = warp_sum(second ? 0.f : qv);
      const float a1 = warp_sum(second ? sv : 0.f), c1 = warp_sum(second ? qv : 0.f);
      if (lane == 0) {
        atomicAdd(&p.st_out[b_first].s, (double)a0);
        atomicAdd(&p.st_out[b_first].ss, (double)c0);
        if (e1 < r0 + nrows) {
          atomicAdd(&p.st_out[b_first + 1].s, (double)a1);
          atomicAdd(&p.st_out[b_first + 1].ss, (double)c1);
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

}  // namespace

cudaError_t conv1_tma_setup() {
  cudaError_t e = cudaFuncSetAttribute(k_conv1_tma<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(k_conv1_tma<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
  return e;
}

void launch_conv1_tma(const Conv1TmaParams& c, cudaStream_t st) {
  TmaParams p{};
  p.a_tmap = *reinterpret_cast<const CUtensorMap*>(c.a_tmap);
  p.M = c.M; p.T = c.T; p.ntiles = (c.M + kTileM - 1) / kTileM; p.Mp = c.Mp;
  p.w_img = c.w_img; p.sb = c.sb; p.st_in = c.norm.gamma ? c.norm.st : nullptr; p.inv_n = c.norm.inv_n; p.eps = c.norm.eps;
  p.slope = c.slope; p.out = c.p_planes; p.st_out = c.st_p;
  const dim3 grid(std::min(ctx().sm_count, p.ntiles));
  if (c.slope <= 1.f) launch_k(k_conv1_tma<true>, grid, dim3(kThreadsT), kSmemBytes, st, true, p);
  else launch_k(k_conv1_tma<false>, grid, dim3(kThreadsT), kSmemBytes, st, true, p);
}

}  // namespace septfa
