// Persistent, warp-specialised tcgen05 kernel for the first contraction of a TCN block (model/model.py:132/138):
//   p = PReLU(W1 GN(stream) + b1),  statistics of p                   (GroupNorm affine folded into W1 / b1)
// One CTA per SM walks 128-frame tiles. In the one-tile-per-CTA kernel (gemm_tc.cu, MODE 0) every CTA alternates a
// read-only phase (load + normalise 128 KB) and a write-only phase (epilogue), and all CTAs of a wave do so in lock
// step, so HBM idles half the time. Here the roles run concurrently on different tiles:
//   warps 0-7   producers : stream rows (fp32) -> (x - mean) * rstd -> fp16 -> 128B-swizzled A stage; the loads of the
//                           next K-chunk - of the NEXT TILE at a tile's end - are always in flight
//   warps 8-11  epilogue  : tcgen05.ld of the previous tile's accumulator (TMEM is double buffered: 2 x 256 columns)
//                           -> +bias, PReLU, statistics, fp16 -> per-warp shared-memory tile -> one TMA bulk store of
//                           a whole row (512 contiguous bytes) per lane
//   warp 12     W loader  : pre-swizzled fp16 weight image chunks by cp.async.bulk (2 stages, L2 resident)
//   warp 13     MMA       : tcgen05.mma 128x256x16, commits release the A / W stages and publish the accumulator
// 14 warps = at most 4 per SM sub-partition, so every thread may use 128 registers (18 warps capped them at 96 and
// spilled the producers' double-buffered loads).
// Synchronisation is mbarriers only (no block barrier inside the tile loop). Requires T >= 128 (a tile then touches at
// most two utterances) and the fp16 activation layout; otherwise launch_tc_conv1 uses the one-tile kernel.
#include <algorithm>
#include <cstdlib>
#include "kernels.h"
#include "tc_common.cuh"

namespace septfa {

namespace {

using namespace tc;

constexpr int kTileM = 128;
constexpr int kNCH = 4;                       // K = 256 = 4 chunks of 64
constexpr int kAStages = 3;
constexpr int kWStages = 2;
constexpr int kABytes = kTileM * 128;         // 16 KB: 128 rows x 64 halves
constexpr int kWBytes = 256 * 128;            // 32 KB: 256 rows x 64 halves
constexpr int kEpiPitch = 512 + 16;           // bytes per staged row (256 fp16 columns + pad: conflict-free STS.128)
constexpr int kEpiWarpBytes = 32 * kEpiPitch; // 16896 B per epilogue warp
constexpr int kOffA = 0;
constexpr int kOffW = kOffA + kAStages * kABytes;
constexpr int kOffEpi = kOffW + kWStages * kWBytes;
constexpr int kOffBias = kOffEpi + 4 * kEpiWarpBytes;   // [256] fp32 bias (broadcast LDS instead of 8 uniform LDG per 32 columns)
constexpr int kOffBar = kOffBias + 1024;
constexpr int kSmemBytes = kOffBar + 256;
// PLANES keeps the weights resident (its epilogue needs no staging buffer): the whole W1 image (4 chunks, 128 KB) is loaded
// once per CTA and stays in shared memory for every tile, so the per-tile traffic into the SM is the A rows only.
constexpr int kAStagesR = 4;
constexpr int kOffWR = kAStagesR * kABytes;                   // 64 KB of A stages, then 128 KB of weights
constexpr int kOffBiasR = kOffWR + kNCH * kWBytes;
constexpr int kOffBarR = kOffBiasR + 1024;
constexpr int kSmemBytesR = kOffBarR + 256;
static_assert(kSmemBytesR <= 232448 && kOffWR % 1024 == 0, "shared-memory plan (resident weights)");
constexpr int kThreadsP = 14 * 32;

struct PersistParams {
  int M, T, ntiles;
  const __half* w_img;
  const float* in;            // [M,256] fp32 stream
  StreamNorm norm;
  const float* bias; float slope;
  __half* out;                // [M,256] fp16, or K-group planes [32][Mp][8] (PLANES)
  int Mp;
  Stat2* st_out;              // [B]
};

// PLANES: p is stored as K-group planes (kernels.h, DconvMmaParams): a lane = a row, so the 32 lanes of a warp write 512
// contiguous bytes per plane straight from registers (full sectors: no staging, no bulk store), and the resident weights
// take the staging buffer's place.
template <bool AMAX, bool PLANES>
__global__ void __launch_bounds__(kThreadsP, 1) k_conv1_persist(PersistParams p) {
  constexpr int kAStages = PLANES ? kAStagesR : septfa::kAStages;
  constexpr int kWStages = PLANES ? kNCH : septfa::kWStages;
  constexpr int kOffW = PLANES ? kOffWR : septfa::kOffW;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (PLANES ? kOffBarR : kOffBar));
  uint64_t* a_full = bars;                    // [kAStages] 256 producer arrivals
  uint64_t* a_empty = bars + 4;               // [kAStages] MMA commit
  uint64_t* w_full = bars + 8;                // [kWStages] bulk copy bytes
  uint64_t* w_empty = bars + 12;              // [2] MMA commit (streaming variant)
  uint64_t* acc_full = bars + 14;             // [2] MMA commit
  uint64_t* acc_empty = bars + 16;            // [2] 128 epilogue arrivals
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 18);
  float* bias_s = reinterpret_cast<float*>(smem + (PLANES ? kOffBiasR : kOffBias));
  constexpr uint32_t IDESC = make_idesc_f16(kTileM, 256);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    if ((smem_u32(smem) & 1023u) != 0u) __trap();
    for (int s = 0; s < kAStages; ++s) { mbar_init(a_full + s, 256); mbar_init(a_empty + s, 1); }
    for (int s = 0; s < kWStages; ++s) mbar_init(w_full + s, 1);
    for (int s = 0; s < 2; ++s) { mbar_init(w_empty + s, 1); mbar_init(acc_full + s, 1); mbar_init(acc_empty + s, 128); }
    fence_mbar_init();
    if constexpr (PLANES) {   // static weights: the whole image, once, before the dependency wait
      for (int j = 0; j < kNCH; ++j) {
        mbar_expect_tx(w_full + j, kWBytes);
        bulk_copy_g2s(smem + kOffW + j * kWBytes, reinterpret_cast<const uint8_t*>(p.w_img) + (size_t)j * kWBytes, kWBytes, w_full + j);
      }
    }
  }
  if (warp == 13) tmem_alloc(tmem_slot, 512);
  if (threadIdx.x < kC) bias_s[threadIdx.x] = __ldg(p.bias + threadIdx.x);   // static weights: before the dependency wait
  pdl_launch_dependents();
  pdl_wait();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int first = blockIdx.x, stride = gridDim.x;

  if (warp < 8) {
    // ------------------------------------------------------------ producers
    const int c8 = lane & 7, rg = lane >> 3;
    const bool has_norm = p.norm.gamma != nullptr;
    float4 xa[2][4], xb[2][4];
    auto issue = [&](int tile, int jj, int buf) {
      const int r0 = tile * kTileM, nrows = min(kTileM, p.M - r0);
#pragma unroll
      for (int it = 0; it < 4; ++it) {
        const int rl = it * 32 + warp * 4 + rg;
        if (rl < nrows) {
          const float4* src = reinterpret_cast<const float4*>(p.in + (int64_t)(r0 + rl) * kC + jj * 64 + c8 * 8);
          xa[buf][it] = __ldg(src);
          xb[buf][it] = __ldg(src + 1);
        } else {
          xa[buf][it] = xb[buf][it] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
    };
    int g = 0;   // chunks produced so far by this CTA
    if (first < p.ntiles) issue(first, 0, 0);
    for (int tile = first; tile < p.ntiles; tile += stride) {
      const int r0 = tile * kTileM, nrows = min(kTileM, p.M - r0);
      const int b_first = r0 / p.T, e1 = (b_first + 1) * p.T;   // first row of the tile's second utterance
      // mean / rstd of the tile's (at most two) utterances: lanes 0 / 1 compute, the warp reads them by shuffle
      float2 mr = make_float2(0.f, 1.f);
      if (has_norm && lane < 2 && (lane == 0 || e1 < r0 + nrows)) mr = stat_mean_rstd(p.norm.st + b_first + lane, p.norm.inv_n, p.norm.eps);
      const float m0 = __shfl_sync(0xffffffffu, mr.x, 0), s0 = __shfl_sync(0xffffffffu, mr.y, 0);
      const float m1 = __shfl_sync(0xffffffffu, mr.x, 1), s1 = __shfl_sync(0xffffffffu, mr.y, 1);
      float sc[4], nb[4];
#pragma unroll
      for (int it = 0; it < 4; ++it) {
        const int rl = it * 32 + warp * 4 + rg;
        const bool second = r0 + rl >= e1;
        const float mean = second ? m1 : m0, rstd = second ? s1 : s0;
        sc[it] = rl < nrows ? rstd : 0.f;
        nb[it] = rl < nrows ? -mean * rstd : 0.f;
      }
#pragma unroll
      for (int j = 0; j < kNCH; ++j, ++g) {
        const int s = g % kAStages, u = g / kAStages;
        // next chunk's loads in flight before this one is converted: the next tile's first chunk at a tile's end
        if (j + 1 < kNCH) issue(tile, j + 1, (j + 1) & 1);
        else if (tile + stride < p.ntiles) issue(tile + stride, 0, 0);
        if (u > 0) mbar_wait(a_empty + s, (u - 1) & 1, 400 + j);
        uint8_t* a_tile = smem + kOffA + s * kABytes;
#pragma unroll
        for (int it = 0; it < 4; ++it) {
          const int rl = it * 32 + warp * 4 + rg;
          const float4 x0 = xa[j & 1][it], x1 = xb[j & 1][it];
          const float k = sc[it], b = nb[it];
          const uint4 pk = make_uint4(pack_half2(fmaf(x0.x, k, b), fmaf(x0.y, k, b)), pack_half2(fmaf(x0.z, k, b), fmaf(x0.w, k, b)),
                                      pack_half2(fmaf(x1.x, k, b), fmaf(x1.y, k, b)), pack_half2(fmaf(x1.z, k, b), fmaf(x1.w, k, b)));
          *reinterpret_cast<uint4*>(a_tile + sw128_offset(rl, c8)) = pk;
        }
        fence_proxy_async();
        mbar_arrive(a_full + s);
      }
    }
  } else if (warp < 12) {
    // ------------------------------------------------------------ epilogue
    const int lq = warp & 3;                                 // TMEM lane quarter (hardware: warp % 4); a lane = a row
    uint8_t* stg = smem + kOffEpi + (warp - 8) * kEpiWarpBytes + lane * kEpiPitch;
    const float2 sl2 = make_float2(p.slope, p.slope);
    int lt = 0;
    for (int tile = first; tile < p.ntiles; tile += stride, ++lt) {
      const int buf = lt & 1;
      const int r0 = tile * kTileM, nrows = min(kTileM, p.M - r0);
      const int b_first = r0 / p.T, e1 = (b_first + 1) * p.T;
      const int rl = lq * 32 + lane;
      const bool valid = rl < nrows;
      mbar_wait(acc_full + buf, (lt >> 1) & 1, 500);
      tc_fence_after();
      if constexpr (!PLANES) bulk_wait_read_all();   // this lane's previous row piece has left the staging buffer
      float2 s2 = make_float2(0.f, 0.f), q2 = make_float2(0.f, 0.f);
#pragma unroll 1
      for (int cc = 0; cc < 8; ++cc) {
        const int col0 = cc * 32;
        float v[32];
        tmem_ld32(tmem_base + (uint32_t)(buf * 256) + ((uint32_t)(lq * 32) << 16) + (uint32_t)col0, v);
        if (cc == 7) {               // the accumulator is in registers: hand the TMEM buffer back to the MMA warp
          tc_fence_before();
          mbar_arrive(acc_empty + buf);
        }
        uint4* dst = reinterpret_cast<uint4*>(stg + cc * 64);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          uint32_t h[4];
#pragma unroll
          for (int k = 0; k < 2; ++k) {
            const int c = 8 * i + 4 * k;
            const float4 b4 = *reinterpret_cast<const float4*>(bias_s + col0 + c);   // same address in every lane: broadcast
            const float2 x0 = __fadd2_rn(make_float2(v[c], v[c + 1]), make_float2(b4.x, b4.y));
            const float2 x1 = __fadd2_rn(make_float2(v[c + 2], v[c + 3]), make_float2(b4.z, b4.w));
            const float2 a0 = __fmul2_rn(sl2, x0), a1 = __fmul2_rn(sl2, x1);
            float2 y0, y1;
            if constexpr (AMAX) { y0 = make_float2(fmaxf(x0.x, a0.x), fmaxf(x0.y, a0.y)); y1 = make_float2(fmaxf(x1.x, a1.x), fmaxf(x1.y, a1.y)); }
            else { y0 = make_float2(fminf(x0.x, a0.x), fminf(x0.y, a0.y)); y1 = make_float2(fminf(x1.x, a1.x), fminf(x1.y, a1.y)); }
            s2 = __fadd2_rn(s2, __fadd2_rn(y0, y1));
            q2 = __ffma2_rn(y0, y0, q2);
            q2 = __ffma2_rn(y1, y1, q2);
            h[2 * k] = pack_half2(y0.x, y0.y);
            h[2 * k + 1] = pack_half2(y1.x, y1.y);
          }
          if constexpr (PLANES) {
            if (valid)
              *reinterpret_cast<uint4*>(p.out + ((size_t)(cc * 4 + i) * p.Mp + (size_t)(kPlaneHalo + r0 + rl)) * 8) =
                  make_uint4(h[0], h[1], h[2], h[3]);
          } else {
            dst[i] = make_uint4(h[0], h[1], h[2], h[3]);
          }
        }
      }
      if constexpr (!PLANES) {
        fence_proxy_async();           // this lane wrote its own row piece: no other lane's data is needed
        if (valid) {
          bulk_copy_s2g(p.out + (int64_t)(r0 + rl) * kC, stg, 512);
          bulk_commit_group();
        }
      }
      // statistics of this warp's 32 rows, per utterance: fixed-order shuffle trees, one double atomic pair
      const bool second = r0 + rl >= e1;
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
    if constexpr (!PLANES) bulk_wait_read_all();
  } else if (warp == 12) {
    // ------------------------------------------------------------ weight loader
    if (!PLANES && lane == 0) {
      int g = 0;
      for (int tile = first; tile < p.ntiles; tile += stride) {
        for (int j = 0; j < kNCH; ++j, ++g) {
          const int s = g % kWStages, u = g / kWStages;
          if (u > 0) mbar_wait(w_empty + s, (u - 1) & 1, 100 + j);
          mbar_expect_tx(w_full + s, kWBytes);
          bulk_copy_g2s(smem + kOffW + s * kWBytes, reinterpret_cast<const uint8_t*>(p.w_img) + (size_t)j * kWBytes, kWBytes, w_full + s);
        }
      }
    }
    __syncwarp();
  } else {
    // ------------------------------------------------------------ MMA issuer
    if (lane == 0) {
      int ga = 0, gw = 0, lt = 0;
      for (int tile = first; tile < p.ntiles; tile += stride, ++lt) {
        const int buf = lt & 1, ub = lt >> 1;
        if (ub > 0) { mbar_wait(acc_empty + buf, (ub - 1) & 1, 600); tc_fence_after(); }
        for (int j = 0; j < kNCH; ++j, ++ga, ++gw) {
          const int sa = ga % kAStages, ua = ga / kAStages, sw = PLANES ? j : gw % kWStages, uw = PLANES ? 0 : gw / kWStages;
          if (!PLANES || lt == 0) mbar_wait(w_full + sw, uw & 1, 200 + j);
          mbar_wait(a_full + sa, ua & 1, 300 + j);
          tc_fence_after();
          const uint64_t a_desc = make_sw128_desc(smem_u32(smem + kOffA + sa * kABytes));
          const uint64_t b_desc = make_sw128_desc(smem_u32(smem + kOffW + sw * kWBytes));
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)
            umma_f16(tmem_base + (uint32_t)(buf * 256), a_desc + (uint64_t)(kk * 2), b_desc + (uint64_t)(kk * 2), IDESC, (j | kk) != 0);
          umma_commit(a_empty + sa);
          if constexpr (!PLANES) umma_commit(w_empty + sw);
        }
        umma_commit(acc_full + buf);
      }
    }
    __syncwarp();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 13) tmem_dealloc(tmem_base, 512);
}

}  // namespace

cudaError_t conv1_persist_setup() {
  cudaError_t e = cudaFuncSetAttribute(k_conv1_persist<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(k_conv1_persist<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(k_conv1_persist<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytesR);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(k_conv1_persist<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytesR);
  return e;
}

void launch_conv1_persist(const Conv1Params& c, cudaStream_t st) {
  PersistParams p{};
  p.M = c.M; p.T = c.T; p.ntiles = (c.M + kTileM - 1) / kTileM;
  p.w_img = c.w_img; p.in = c.w_in; p.norm = c.norm; p.bias = c.bias_f; p.slope = c.slope;
  p.out = reinterpret_cast<__half*>(c.p_out); p.st_out = c.st_p; p.Mp = c.Mp;
  const dim3 grid(std::min(ctx().sm_count, p.ntiles));
  if (c.planes) {
    if (c.slope <= 1.f) launch_k(k_conv1_persist<true, true>, grid, dim3(kThreadsP), kSmemBytesR, st, true, p);
    else launch_k(k_conv1_persist<false, true>, grid, dim3(kThreadsP), kSmemBytesR, st, true, p);
  } else {
    if (c.slope <= 1.f) launch_k(k_conv1_persist<true, false>, grid, dim3(kThreadsP), kSmemBytes, st, true, p);
    else launch_k(k_conv1_persist<false, false>, grid, dim3(kThreadsP), kSmemBytes, st, true, p);
  }
}

}  // namespace septfa
