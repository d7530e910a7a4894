// TMA-fed, CTA-pair (cta_group::2) TF32 tcgen05 kernel for the first contraction of a TCN block (model/model.py:132/138),
// blocks 1 .. n-1 of the recursive-LN wiring in the fast precision mode:
//   p = PReLU(W1 GN(stream) + b1),  statistics of p
// The persistent kernel of gemm_conv1_persist.cu spends its time in eight producer warps (fp32 rows -> normalise -> fp16
// -> swizzled shared memory, one K-chunk of loads in flight per thread: ~3 k cycles per chunk of pure latency). Here no
// thread touches the A operand: the fp32 residual stream is the operand itself,
//   W' ((w - mean) rstd) + b' = rstd (W' w) + (b' - rstd mean S),   W' = W1 diag(gamma),  S[n] = sum_k W'[n,k],
// fetched by TMA tensor loads (box 32 floats x 128 rows, 128-byte swizzle = the K-major SWIZZLE_128B operand layout) and
// multiplied as TF32 (kind::tf32: the tensor core reads the upper 19 bits of each fp32, 11 significant bits like fp16).
// The weights are TF32 too (rounded to nearest on the host), 256 KB - so the CTAs run as PAIRS: every MMA is a
// tcgen05.mma.cta_group::2 of M = 256 (128 frames per CTA) whose B operand is split along N between the two CTAs, and
// each CTA keeps its half of the image (128 KB) resident in shared memory for the whole kernel. Per 128-frame tile an SM
// takes in the tile's 128 KB of stream and nothing else.
// Roles per CTA (12 warps):
//   warp 0       TMA producer : ring of 5 A stages (16 KB = one K-chunk of 32 of this CTA's tile), runs ahead across tiles
//   warp 1       MMA issuer (leader CTA): per K-chunk 4 MMAs (M256 N256 K8), double-buffered accumulator (2 x 256 TMEM columns per
//                CTA); commits are multicast to both CTAs
//   warp 2       static loader (prologue): this CTA's half of the weight image
//   warp 3       relay (peer CTA): forwards "my A stage / my weights have landed" to the leader's barriers
//   warps 4-11   epilogue     : tcgen05.ld -> rstd * acc + (b' - rstd mean S) -> PReLU -> statistics -> fp16 -> K-group planes
//                of p (kernels.h, DconvMmaParams); a lane = a row, 32 lanes = 512 contiguous bytes per plane
// Requires T >= 128 (a tile touches at most two utterances).
#include <algorithm>
#include <cuda.h>
#include "kernels.h"
#include "tc_common.cuh"

namespace septfa {

namespace {

using namespace tc;

constexpr int kTileM = 128;
constexpr int kNCH = 8;                       // K = 256 = 8 chunks of 32 floats
constexpr int kAStages = 5;
constexpr int kABytes = kTileM * 128;         // 16 KB: 128 rows x 32 floats
constexpr int kWHalfBytes = 128 * 128;        // 16 KB: this CTA's 128 output rows of one K-chunk
constexpr int kOffA = 0;
constexpr int kOffW = kOffA + kAStages * kABytes;            // 80 KB
constexpr int kOffSb = kOffW + kNCH * kWHalfBytes;           // + 128 KB
constexpr int kOffBar = kOffSb + 2048;
constexpr int kSmemBytes = kOffBar + 512;
constexpr int kEpiWarps = 8;                  // 4 TMEM lane quarters x 2 column halves
constexpr int kEpiCols = 256 / (kEpiWarps / 4);
constexpr int kThreadsC = (4 + kEpiWarps) * 32;
static_assert(kOffW % 1024 == 0 && kSmemBytes <= 232448, "shared-memory plan");

struct PairParams {
  alignas(64) CUtensorMap a_tmap;   // the stream: fp32 [M rows][256], box 32 x 128, SWIZZLE_128B
  int M, T, ntiles, Mp;
  const float* w_img;               // TF32 image: 8 K-chunks x [256 rows x 128 B], 128B-swizzled K-major
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
__device__ __forceinline__ void tmem_alloc2(uint32_t* slot, uint32_t ncols) {   // one warp of EACH CTA of the pair, same slot offset
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem, 256 rows over the pair] (+)= A[smem of each CTA: its 128 rows] * B[smem of each CTA: its half of N]^T, TF32 operands
__device__ __forceinline__ void umma2_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(0u)
      : "memory");
}
__device__ __forceinline__ void umma2_commit(uint64_t* bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
               "h"(mask)
               : "memory");
}
// Arrive on the barrier at this offset in CTA `rank` of the cluster (CTA-scope semantics, see dconv_mma2.cu).
__device__ __forceinline__ void mbar_arrive_cl(uint64_t* bar, uint32_t rank) {
  uint32_t remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(bar)), "r"(rank));
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
}
// Instruction descriptor: D = F32 [4,6) = 1, A = TF32 [7,10) = 2, B = TF32 [10,13) = 2, K-major, N >> 3 [17,23), M >> 4 [24,29)
__host__ __device__ constexpr uint32_t make_idesc_tf32(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

template <bool AMAX>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreadsC, 1) k_conv1_pair(const __grid_constant__ PairParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kOffBar);
  uint64_t* a_full = bars;                    // [5] TMA bytes
  uint64_t* a_peer = bars + 5;                // [5] leader: the peer's stage has landed (relay)
  uint64_t* a_empty = bars + 10;              // [5] MMA commit (multicast)
  uint64_t* w_full = bars + 15;               // [8] bulk copy bytes (once)
  uint64_t* w_peer = bars + 23;               // [8] leader: relay
  uint64_t* acc_full = bars + 31;             // [2] MMA commit (multicast)
  uint64_t* acc_empty = bars + 33;            // [2] leader: 16 epilogue warps of the pair
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 36);
  const float4* sb_s = reinterpret_cast<const float4*>(smem + kOffSb);
  constexpr uint32_t IDESC = make_idesc_tf32(2 * kTileM, 256);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t crank = cluster_ctarank();
  const bool leader = crank == 0;
  if (threadIdx.x == 0) {
    if ((smem_u32(smem) & 1023u) != 0u) __trap();
    for (int s = 0; s < kAStages; ++s) { mbar_init(a_full + s, 1); mbar_init(a_peer + s, 1); mbar_init(a_empty + s, 1); }
    for (int j = 0; j < kNCH; ++j) { mbar_init(w_full + j, 1); mbar_init(w_peer + j, 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(acc_full + s, 1); mbar_init(acc_empty + s, 2 * kEpiWarps); }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc2(tmem_slot, 512);
  if (threadIdx.x < 128) reinterpret_cast<float4*>(smem + kOffSb)[threadIdx.x] = __ldg(p.sb + threadIdx.x);
  __syncthreads();
  if (warp == 2 && lane == 0) {
    // static weights, once, before the dependency wait: rows 128 r .. 128 r + 127 of every K-chunk (16 KB contiguous)
    for (int j = 0; j < kNCH; ++j) {
      mbar_expect_tx(w_full + j, kWHalfBytes);
      bulk_copy_g2s(smem + kOffW + j * kWHalfBytes, reinterpret_cast<const uint8_t*>(p.w_img) + (size_t)j * 2 * kWHalfBytes + (size_t)crank * kWHalfBytes,
                    kWHalfBytes, w_full + j);
    }
  }
  pdl_launch_dependents();
  pdl_wait();
  tc_fence_before();
  cluster_sync_all();   // (also a CTA barrier) both CTAs' mbarriers are initialised and their tensor memory is allocated
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // the pair walks tile pairs: cluster c takes pairs c, c + nclusters, ...; rank r the tile 2 * pair + r (an odd tile count
  // leaves the last pair with an empty tile: its rows read as zeros and nothing is stored)
  const int npairs = (p.ntiles + 1) / 2;
  const int first_pair = (int)blockIdx.x / 2, pair_stride = (int)gridDim.x / 2;
  const int my_tiles = first_pair < npairs ? (npairs - first_pair + pair_stride - 1) / pair_stride : 0;
  const int first = 2 * first_pair + (int)crank, stride = 2 * pair_stride, tile_end = 2 * npairs;

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer (rows past M read as zeros)
    if (lane == 0) {
      int g = 0;
      for (int tile = first; tile < tile_end; tile += stride) {
        for (int j = 0; j < kNCH; ++j, ++g) {
          const int s = g % kAStages, u = g / kAStages;
          if (u > 0) mbar_wait(a_empty + s, (u - 1) & 1, 100 + j);
          mbar_expect_tx(a_full + s, kABytes);
          tma_load_2d(smem + kOffA + s * kABytes, &p.a_tmap, j * 32, tile * kTileM, a_full + s);
        }
      }
    }
    __syncwarp();
  } else if (warp == 3) {
    // ------------------------------------------------------------ relay (peer CTA): tell the leader what has landed here
    if (!leader && lane == 0) {
      const int total = my_tiles * kNCH;
      for (int g = 0; g < max(total, kNCH); ++g) {
        if (g < kNCH) { mbar_wait(w_full + g, 0, 170 + g); mbar_arrive_cl(w_peer + g, 0); }
        if (g < total) {
          const int s = g % kAStages, u = g / kAStages;
          mbar_wait(a_full + s, u & 1, 180);
          mbar_arrive_cl(a_peer + s, 0);
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer (leader CTA)
    if (leader && lane == 0) {
      int g = 0;
      for (int lt = 0; lt < my_tiles; ++lt) {
        const int buf = lt & 1, ub = lt >> 1;
        if (ub > 0) { mbar_wait(acc_empty + buf, (ub - 1) & 1, 600); tc_fence_after(); }
        for (int j = 0; j < kNCH; ++j, ++g) {
          const int sa = g % kAStages, ua = g / kAStages;
          if (lt == 0) { mbar_wait(w_full + j, 0, 200 + j); mbar_wait(w_peer + j, 0, 210 + j); }
          mbar_wait(a_full + sa, ua & 1, 300 + j);
          mbar_wait(a_peer + sa, ua & 1, 310 + j);
          tc_fence_after();
          const uint64_t a_desc = make_sw128_desc(smem_u32(smem + kOffA + sa * kABytes));
          const uint64_t b_desc = make_sw128_desc(smem_u32(smem + kOffW + j * kWHalfBytes));
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)   // K = 8 floats = 32 bytes per MMA
            umma2_tf32(tmem_base + (uint32_t)(buf * 256), a_desc + (uint64_t)(kk * 2), b_desc + (uint64_t)(kk * 2), IDESC, (j | kk) != 0);
          umma2_commit(a_empty + sa, (uint16_t)3);
        }
        umma2_commit(acc_full + buf, (uint16_t)3);
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
    for (int tile = first; tile < tile_end; tile += stride, ++lt) {
      const int buf = lt & 1;
      const int r0 = tile * kTileM, nrows = max(0, min(kTileM, p.M - r0));
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
      // two tensor-memory loads in flight; the next tile's statistics are computed under the first pair
      constexpr int NC = kEpiCols / 32;
      uint32_t va[32], vb[32];
      tmem_ld32_nowait(t_row, va);
      tmem_ld32_nowait(t_row + 32u, vb);
      mr = tile_stats(tile + stride);
#pragma unroll
      for (int c2 = 0; c2 < NC / 2; ++c2) {
        tmem_ld_wait();                // va and vb (chunks 2 c2, 2 c2 + 1) have landed
        if (c2 + 1 == NC / 2) {        // this warp's part of the accumulator is in registers: one arrival per warp, on the leader's barrier
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_cl(acc_empty + buf, 0);
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
      if (lane == 0 && nrows > 0) {
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
  cluster_sync_all();   // neither CTA leaves (or frees its tensor memory) while the pair's MMAs may still touch it
  if (warp == 1) tmem_dealloc2(tmem_base, 512);
}

}  // namespace

cudaError_t conv1_pair_setup() {
  cudaError_t e = cudaFuncSetAttribute(k_conv1_pair<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(k_conv1_pair<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
  return e;
}

void launch_conv1_pair(const Conv1PairParams& c, cudaStream_t st) {
  PairParams p{};
  p.a_tmap = *reinterpret_cast<const CUtensorMap*>(c.a_tmap);
  p.M = c.M; p.T = c.T; p.ntiles = (c.M + kTileM - 1) / kTileM; p.Mp = c.Mp;
  p.w_img = c.w_img; p.sb = c.sb; p.st_in = c.norm.gamma ? c.norm.st : nullptr; p.inv_n = c.norm.inv_n; p.eps = c.norm.eps;
  p.slope = c.slope; p.out = c.p_planes; p.st_out = c.st_p;
  const int npairs = (p.ntiles + 1) / 2;
  const dim3 grid(2 * std::min(ctx().sm_count / 2, npairs));
  if (c.slope <= 1.f) launch_k(k_conv1_pair<true>, grid, dim3(kThreadsC), kSmemBytes, st, true, p);
  else launch_k(k_conv1_pair<false>, grid, dim3(kThreadsC), kSmemBytes, st, true, p);
}

}  // namespace septfa
