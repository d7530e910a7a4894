// tcgen05 engine for the three dense contractions of the TCN (the 1x1 convolutions):
//   MODE 0  conv1d      256 -> 256 : A = GN(stream) computed on load;  epilogue +bias, PReLU, stats
//   MODE 1  dconv+conv3 512 -> 256 : A = PReLU(depthwise-dilated-conv(GN1(p))) computed on load
//                                    (q never leaves the SM); epilogue raw accumulators + row/col sums
//   MODE 2  output conv 256 -> 514 : A = GN(PReLU(GN(stream))) on load; epilogue +bias
// One CTA = one 128-frame tile (UMMA M = 128, cta_group::1) x one N tile (256, or 192 x 3 for MODE 2).
// fp16 operands in shared memory (K-major, 128-byte swizzle), fp32 accumulators in TMEM.
//   warps 0-7 : produce the A operand chunk by chunk (global fp32 -> transform -> fp16 -> swizzled
//               st.shared), then run the epilogue (tcgen05.ld -> shared staging -> coalesced stores)
//   warp 8    : streams the pre-swizzled weight image with cp.async.bulk (TMA bulk copy) + mbarrier
//   warp 9    : allocates TMEM, issues tcgen05.mma (one elected thread), tcgen05.commit -> mbarriers
// Reference semantics: model/model.py:130-149 (DepthConv1d), :322-325,357 (TCN.output).
#include <cstdio>
#include <cstdlib>
#include <type_traits>
#include "kernels.h"
#include "tc_common.cuh"

namespace septfa {

namespace {

constexpr int kTileM = 128;
constexpr int kAChunkBytes = kTileM * 128;  // one K-chunk (64 halves = 128 B) of the A tile
constexpr int kStages = 2;
constexpr int kThreads = 320;
constexpr int kAuxBytes = 4096;
constexpr int kDconvWBytes = 2 * 256 * 16 + 256 * 8;  // MODE 1: folded depthwise taps staged in shared memory (10 KB)
constexpr int kStgPitch = 36;               // floats per staged row (32 + 4 pad, 16 B aligned)

struct TcParams {
  int M, T, B;
  const __half* w_img;
  const __half* w_img_lo;   // MODE 2 / SPLIT: low part of the fp16 split of the weights
  const void* in;           // [M,256] fp32 (MODE 0/2, and MODE 1 when !H16) or fp16 (MODE 1 with H16)
  StreamNorm norm;
  // MODE 2 prologue
  float slope_o; const Stat2* st_o; const float* g_o; const float* b_o;
  // MODE 1 prologue
  const Stat2* st_p; const float4* wtab; const float* bog;
  float slope2; int dil; Stat2* st_q;
  // epilogue
  const float* bias; float slope;
  void* out; int out_stride;  // fp32, or fp16 for MODE 0/1 with H16
  Stat2* st_out;
  float* rowsum; double* colsum;
};

using namespace tc;

__device__ __forceinline__ float4 ld_half4(const __half* p) {   // 4 consecutive halves (8 B) -> float4
  const uint2 v = __ldg(reinterpret_cast<const uint2*>(p));
  const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&v.x));
  const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&v.y));
  return make_float4(a.x, a.y, b.x, b.y);
}

// Low part of the 2-term fp16 split: fp16(x - fp16(x)), the residual being exact in fp32.
__device__ __forceinline__ uint32_t pack_residual2(float a, float b, uint32_t hi) {
  const float2 h = __half22float2(*reinterpret_cast<const __half2*>(&hi));
  return pack_half2(a - h.x, b - h.y);
}
__device__ __forceinline__ uint4 pack_residual8(const float (&y)[8], const uint4& hi) {
  return make_uint4(pack_residual2(y[0], y[1], hi.x), pack_residual2(y[2], y[3], hi.y), pack_residual2(y[4], y[5], hi.z),
                    pack_residual2(y[6], y[7], hi.w));
}

// H16: the activation tensor exchanged with the neighbouring contraction (conv1's output p = dconv's input; dconv's
// output racc) is stored as fp16 instead of fp32.
// AMAX (MODE 1): the PReLU slope of the depthwise stage is <= 1, so PReLU(x) = max(x, a x); otherwise min(x, a x).
// SPLIT (MODE 0 / 1): split-precision operands - A = A_hi + A_lo and W = W_hi + W_lo, each part fp16, three tensor-core
// passes A_hi W_hi + A_lo W_hi + A_hi W_lo into the same fp32 accumulator (the A_lo W_lo term is below 2^-22 relative):
// the contraction is then fp32-accurate. Used with fp32 storage of p / racc (H16 = false) by the "accurate" precision
// mode, which config_without_vad needs (its un-renormalised residual stream accumulates the fp16 rounding of every
// block: DESIGN.md, "Precision"). The stage then holds [A_hi][A_lo][W_hi][W_lo] = 96 KB: one CTA per SM.
template <int MODE, bool H16, bool AMAX = true, bool SPLIT = false>
__global__ void __launch_bounds__(kThreads, SPLIT ? 1 : 2) k_tc_gemm(TcParams p) {
  constexpr int NT = (MODE == 2) ? 192 : 256;
  constexpr int KDIM = (MODE == 1) ? 512 : 256;
  constexpr int NCH = KDIM / 64;
  constexpr int WCH = NT * 128;
  // MODE 2 runs a 3-pass fp16 split (A = A_hi + A_lo, W = W_hi + W_lo; A_hi W_hi + A_lo W_hi + A_hi W_lo): the output
  // conv feeds the VAD head directly and dominated its error budget, and costs < 3 % of the FLOPs.
  constexpr int NSPLIT = (MODE == 2 || SPLIT) ? 2 : 1;
  constexpr int STAGE = NSPLIT * (kAChunkBytes + WCH);   // [A_hi][A_lo][W_hi][W_lo]
  constexpr int OFF_W = NSPLIT * kAChunkBytes;
  constexpr uint32_t IDESC = make_idesc_f16(kTileM, NT);

  // 1024-byte alignment for the 128B swizzle. The kernel has no static shared memory, so the dynamic window starts at
  // the CTA's (1 KB aligned) shared base; declaring the alignment lets every shared address be a compile-time offset
  // from one base register (a run-time round-up was re-derived inside the producer loop under register pressure:
  // S2UR CgaCtaId / LOP3 0x3f0 / IMAD chains in every chunk). Checked once instead of corrected.
  extern __shared__ __align__(1024) uint8_t smem[];
  if (threadIdx.x == 0 && (smem_u32(smem) & 1023u) != 0u) __trap();
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kStages * STAGE);
  uint64_t* full_a = bars;          // [kStages] producers -> MMA
  uint64_t* full_w = bars + 2;      // [kStages] bulk copy -> MMA
  uint64_t* empty = bars + 4;       // [kStages] MMA -> producers / loader
  uint64_t* acc_full = bars + 6;    // MMA -> epilogue
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 7);
  float2* tab_a = reinterpret_cast<float2*>(bars + 8);
  float2* tab_b = tab_a + kMaxSegs;
  float* seg_acc = reinterpret_cast<float*>(tab_b + kMaxSegs);
  float* rs_x = seg_acc + 2 * kMaxSegs;  // [128] row-sum exchange between the two column halves
  float* slots = rs_x + kTileM;          // [8 warps][4] per-warp statistics partials
  // MODE 1: folded depthwise taps in pair order, [chunk 8][pair 4][c8 8] each (pack_dconv_taps)
  float4* wA_s = reinterpret_cast<float4*>(reinterpret_cast<uint8_t*>(bars) + kAuxBytes);   // {wx_a, wx_b, wy_a, wy_b}
  float4* wB_s = wA_s + 256;                                                                  // {wz_a, wz_b, sw_a, sw_b}
  float2* wC_s = reinterpret_cast<float2*>(wB_s + 256);                                       // {c2f_a, c2f_b}

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // MODE 2 (three N-tiles per M-tile): a 1-D grid with the N-tile index fastest, so that the three CTAs that read the
  // same 128 rows of the stream run next to each other and the second and third read hit the L2 (with the M-tile index
  // fastest the stream came from HBM three times: 180 MB read per launch against 66 MB)
  const int bx = (MODE == 2) ? (int)blockIdx.x / 3 : (int)blockIdx.x;
  const int by = (MODE == 2) ? (int)blockIdx.x % 3 : (int)blockIdx.y;
  const int r0 = bx * kTileM;
  const int nrows = min(kTileM, p.M - r0);
  const SegMap smap(r0, p.T);
  const int b_first = smap.b_first;
  const int nseg = (r0 + nrows - 1) / p.T - b_first + 1;
  const __half* w_img = p.w_img + (size_t)by * NCH * (WCH / 2);
  const __half* w_img_lo = (NSPLIT == 2) ? p.w_img_lo + (size_t)by * NCH * (WCH / 2) : nullptr;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(full_a + s, 256);
      mbar_init(full_w + s, 1);
      mbar_init(empty + s, 1);
    }
    mbar_init(acc_full, 1);
    fence_mbar_init();
  }
  if (warp == 9) tmem_alloc(tmem_slot, 256);
  // MODE 1 (dconv) does not trigger its dependents: its successor is a persistent grid, which must not take SM slots
  // this grid's second wave still needs (resid_fused.cu)
  if (MODE != 1) pdl_launch_dependents();
  if (MODE == 1) {
    // folded depthwise taps (static weights): staged before waiting for the previous kernel; the global image already
    // has the shared-memory layout (consecutive c8 = consecutive 16 B: conflict-free LDS.128 across a warp)
    for (int i = threadIdx.x; i < kDconvWBytes / 16; i += kThreads) wA_s[i] = __ldg(p.wtab + i);
  }
  pdl_wait();   // everything below reads what earlier kernels of the chain wrote
  {
    const double inv_n = 1.0 / ((double)kC * p.T);
    for (int i = threadIdx.x; i < nseg; i += kThreads) {
      if (MODE == 1) {
        const float2 mr = stat_mean_rstd(p.st_p + b_first + i, inv_n, 1e-8f);
        tab_a[i] = mr;
        tab_b[i] = make_float2(mr.x, 1.0f / mr.y);   // (mean, 1 / rstd): the input value that normalises to zero
      } else {
        tab_a[i] = p.norm.gamma != nullptr ? stat_mean_rstd(p.norm.st + b_first + i, p.norm.inv_n, p.norm.eps)
                                           : make_float2(0.f, 1.f);
        if (MODE == 2) tab_b[i] = stat_mean_rstd(p.st_o + b_first + i, inv_n, 1e-5f);
      }
    }
    for (int i = threadIdx.x; i < 2 * nseg; i += kThreads) seg_acc[i] = 0.f;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 8) {
    // ------------------------------------------------------------ weight loader (TMA bulk copies)
    if (lane == 0) {
      for (int j = 0; j < NCH; ++j) {
        const int s = j % kStages, u = j / kStages;
        if (u > 0) mbar_wait(empty + s, (u - 1) & 1, 100 + j);
        mbar_expect_tx(full_w + s, NSPLIT * WCH);
        bulk_copy_g2s(smem + s * STAGE + OFF_W, reinterpret_cast<const uint8_t*>(w_img) + (size_t)j * WCH, WCH, full_w + s);
        if (NSPLIT == 2)
          bulk_copy_g2s(smem + s * STAGE + OFF_W + WCH, reinterpret_cast<const uint8_t*>(w_img_lo) + (size_t)j * WCH, WCH,
                        full_w + s);
      }
    }
    __syncwarp();
  } else if (warp == 9) {
    // ------------------------------------------------------------ MMA issuer
    if (lane == 0) {
      for (int j = 0; j < NCH; ++j) {
        const int s = j % kStages, u = j / kStages;
        mbar_wait(full_w + s, u & 1, 200 + j);
        mbar_wait(full_a + s, u & 1, 300 + j);
        tc_fence_after();
        const uint64_t a_desc = make_sw128_desc(smem_u32(smem + s * STAGE));
        const uint64_t b_desc = make_sw128_desc(smem_u32(smem + s * STAGE + OFF_W));
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {  // UMMA_K = 16 halves = 32 B -> +2 in the (addr >> 4) field
          umma_f16(tmem_base, a_desc + (uint64_t)(kk * 2), b_desc + (uint64_t)(kk * 2), IDESC, (j | kk) != 0);
          if (NSPLIT == 2) {
            const uint64_t a_lo = make_sw128_desc(smem_u32(smem + s * STAGE + kAChunkBytes));
            const uint64_t b_lo = make_sw128_desc(smem_u32(smem + s * STAGE + OFF_W + WCH));
            umma_f16(tmem_base, a_lo + (uint64_t)(kk * 2), b_desc + (uint64_t)(kk * 2), IDESC, 1u);
            umma_f16(tmem_base, a_desc + (uint64_t)(kk * 2), b_lo + (uint64_t)(kk * 2), IDESC, 1u);
          }
        }
        umma_commit(empty + s);
      }
      umma_commit(acc_full);
    }
    __syncwarp();
  } else {
    // ------------------------------------------------------------ A-operand producers (warps 0-7)
    // lane -> (row group rg = lane/8, 16-byte chunk c8 = lane%8); each warp covers 4 rows per step.
    const int c8 = lane & 7, rg = lane >> 3;
    SegStat2 qstat;
    if (MODE == 0) {
      // conv1: A = (x - mean) * rstd (gamma / beta live in the weight image and the bias). The global loads of
      // chunk j+1 are issued before chunk j is converted, so one round trip to HBM is exposed per tile, not per chunk.
      float4 xa[2][4], xb[2][4];
      auto issue = [&](int jj, int buf) {
#pragma unroll
        for (int it = 0; it < 4; ++it) {
          const int rl = it * 32 + warp * 4 + rg;
          if (rl < nrows) {
            const float4* src = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p.in) + (int64_t)(r0 + rl) * kC + jj * 64 + c8 * 8);
            xa[buf][it] = __ldg(src);
            xb[buf][it] = __ldg(src + 1);
          } else {
            xa[buf][it] = xb[buf][it] = make_float4(0.f, 0.f, 0.f, 0.f);
          }
        }
      };
      float2 mrs[4];
#pragma unroll
      for (int it = 0; it < 4; ++it) {
        const int rl = it * 32 + warp * 4 + rg;
        mrs[it] = rl < nrows ? tab_a[smap.seg(r0 + rl)] : make_float2(0.f, 0.f);
      }
      issue(0, 0);
#pragma unroll
      for (int j = 0; j < NCH; ++j) {
        const int s = j % kStages, u = j / kStages;
        if (j + 1 < NCH) issue(j + 1, (j + 1) & 1);
        if (u > 0) mbar_wait(empty + s, (u - 1) & 1, 400 + j);
        uint8_t* a_tile = smem + s * STAGE;
#pragma unroll
        for (int it = 0; it < 4; ++it) {
          const int rl = it * 32 + warp * 4 + rg;
          const float4 x0 = xa[j & 1][it], x1 = xb[j & 1][it];
          const float sc = mrs[it].y, nb = -mrs[it].x * mrs[it].y;
          const float y[8] = {fmaf(x0.x, sc, nb), fmaf(x0.y, sc, nb), fmaf(x0.z, sc, nb), fmaf(x0.w, sc, nb),
                              fmaf(x1.x, sc, nb), fmaf(x1.y, sc, nb), fmaf(x1.z, sc, nb), fmaf(x1.w, sc, nb)};
          const uint4 pk = make_uint4(pack_half2(y[0], y[1]), pack_half2(y[2], y[3]), pack_half2(y[4], y[5]), pack_half2(y[6], y[7]));
          *reinterpret_cast<uint4*>(a_tile + sw128_offset(rl, c8)) = pk;
          if constexpr (NSPLIT == 2) *reinterpret_cast<uint4*>(a_tile + kAChunkBytes + sw128_offset(rl, c8)) = pack_residual8(y, pk);
        }
        fence_proxy_async();
        mbar_arrive(full_a + s);
      }
    } else if (MODE == 1) {
      // dconv + res_out: q channels 64j + 8*c8 .. +7  <-  in-channels g0 .. g0+3 (out-channel o reads in-channel o/2).
      // GroupNorm reg1 is folded into the taps (w2f = w * gamma, sw = sum_k w2f, c2f = b2 + beta * sum_k w):
      //   q = PReLU(rstd * sum_k w2f[k] p[t+(k-1)d] + (c2f - rstd * mean * sw))
      // evaluated on PAIRS of outputs with the packed fp32 pipe (FFMA2): a pair is the two outputs of equal parity of
      // two neighbouring input channels, so its three taps multiply the float2 that one half2 -> float2 conversion of
      // the input yields; the tap table is staged in that pair order (see pack_dconv_taps in septfa_abi.cu).
      // PReLU is max(x, a x) for a <= 1 (min for a > 1): exact, no predicate.
      // Zero padding: the reference pads the NORMALISED signal, so a tap outside the utterance must contribute 0. The
      // folded formula gives exactly that when the missing input is replaced by the value that normalises to zero,
      // p0[c] = mean - (beta[c] / gamma[c]) / rstd - one FFMA2 per channel pair and no separate code path for the
      // frames within `dil` of an utterance edge (a quarter of all rows at these dilations).
      // The global loads of step st+1 (two rows of the next half chunk) are issued before step st is computed.
      using RawT = typename std::conditional<H16, uint2, float4>::type;
      struct Step { RawT xm[2], xc[2], xp[2]; };
      auto ldraw = [](const void* base, int64_t off) -> RawT {
        if constexpr (H16) return __ldg(reinterpret_cast<const uint2*>(reinterpret_cast<const __half*>(base) + off));
        else return __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(base) + off));
      };
      auto to_pairs = [](const RawT& v, float2 (&o)[2]) {
        if constexpr (H16) {
          o[0] = __half22float2(*reinterpret_cast<const __half2*>(&v.x));
          o[1] = __half22float2(*reinterpret_cast<const __half2*>(&v.y));
        } else {
          o[0] = make_float2(v.x, v.y);
          o[1] = make_float2(v.z, v.w);
        }
      };
      // the four rows this lane owns in every chunk: segment | (t-d) inside << 8 | (t+d) inside << 9 | row valid << 10
      int rflag[4];
#pragma unroll
      for (int it = 0; it < 4; ++it) {
        const int rl = it * 32 + warp * 4 + rg;
        rflag[it] = 0;
        if (rl < nrows) {
          const int row = r0 + rl, sg = smap.seg(row), t = smap.frame(row, sg);
          rflag[it] = sg | 1024 | (t - p.dil >= 0 ? 256 : 0) | (t + p.dil < p.T ? 512 : 0);
        }
      }
      const int64_t lane_off = (int64_t)(r0 + warp * 4 + rg) * kC + c8 * 4;   // element offset of row it = 0, chunk 0
      const int dil_off = p.dil * kC;
      const float2 slope2 = make_float2(p.slope2, p.slope2);
      // statistics of q per row slot (a lane owns the same four rows in every chunk); routed to the utterance
      // accumulators once per tile. Rows past the end of the tensor run through the arithmetic like any other (their
      // inputs read as zero; row m of A only reaches row m of the accumulator, which the epilogue never stores) and are
      // dropped here.
      float2 accS[4], accQ[4];
#pragma unroll
      for (int it = 0; it < 4; ++it) accS[it] = accQ[it] = make_float2(0.f, 0.f);
      RawT zero_raw;
      if constexpr (H16) zero_raw = make_uint2(0u, 0u); else zero_raw = make_float4(0.f, 0.f, 0.f, 0.f);

      auto issue = [&](int jj, int half, Step& sp) {
#pragma unroll
        for (int i2 = 0; i2 < 2; ++i2) {
          const int f = half ? rflag[2 + i2] : rflag[i2];
          const int64_t off = lane_off + ((half * 2 + i2) * 32 * kC + jj * 32);
          sp.xc[i2] = (f & 1024) ? ldraw(p.in, off) : zero_raw;
          sp.xm[i2] = (f & 256) ? ldraw(p.in, off - dil_off) : zero_raw;
          sp.xp[i2] = (f & 512) ? ldraw(p.in, off + dil_off) : zero_raw;
        }
      };
      auto compute = [&](int jj, int half, const Step& sp) {
        uint8_t* a_tile = smem + (jj % kStages) * STAGE;
        const float4* WA = wA_s + jj * 32 + c8;   // [chunk][pair][c8]: {wx_a, wx_b, wy_a, wy_b}
        const float4* WB = wB_s + jj * 32 + c8;   //                    {wz_a, wz_b, sw_a, sw_b}
        const float2* WC = wC_s + jj * 32 + c8;   //                    {c2f_a, c2f_b}
        float2 vm[2][2], vc[2][2], vp[2][2], rs2[2], nr2[2];
#pragma unroll
        for (int i2 = 0; i2 < 2; ++i2) {
          const int f = half ? rflag[2 + i2] : rflag[i2];
          const float2 mr = tab_a[f & 255];
          const float nr = -mr.x * mr.y;
          rs2[i2] = make_float2(mr.y, mr.y);
          nr2[i2] = make_float2(nr, nr);
          to_pairs(sp.xc[i2], vc[i2]);
          to_pairs(sp.xm[i2], vm[i2]);
          to_pairs(sp.xp[i2], vp[i2]);
          if ((f & 768) != 768) {   // a tap outside the utterance: substitute the input that normalises to zero
            const float2 mi = tab_b[f & 255];   // (mean, 1 / rstd)
            const float4 bg = __ldg(reinterpret_cast<const float4*>(p.bog + jj * 32 + c8 * 4));
            const float2 ni = make_float2(-mi.y, -mi.y), mm = make_float2(mi.x, mi.x);
            const float2 pad0 = __ffma2_rn(ni, make_float2(bg.x, bg.y), mm), pad1 = __ffma2_rn(ni, make_float2(bg.z, bg.w), mm);
            if (!(f & 256)) { vm[i2][0] = pad0; vm[i2][1] = pad1; }
            if (!(f & 512)) { vp[i2][0] = pad0; vp[i2][1] = pad1; }
          }
        }
        uint32_t pk[2][4];
        [[maybe_unused]] uint32_t pl[2][4];
#pragma unroll
        for (int gp = 0; gp < 2; ++gp) {
          float2 P[2][2];
#pragma unroll
          for (int par = 0; par < 2; ++par) {
            const float4 wa = WA[(gp * 2 + par) * 8], wb = WB[(gp * 2 + par) * 8];
            const float2 cc = WC[(gp * 2 + par) * 8];
#pragma unroll
            for (int i2 = 0; i2 < 2; ++i2) {
              float2 conv = __fmul2_rn(make_float2(wa.x, wa.y), vm[i2][gp]);
              conv = __ffma2_rn(make_float2(wa.z, wa.w), vc[i2][gp], conv);
              conv = __ffma2_rn(make_float2(wb.x, wb.y), vp[i2][gp], conv);
              const float2 k0 = __ffma2_rn(nr2[i2], make_float2(wb.z, wb.w), cc);
              const float2 x = __ffma2_rn(rs2[i2], conv, k0);
              const float2 ax = __fmul2_rn(slope2, x);
              float2 q;
              if constexpr (AMAX) q = make_float2(fmaxf(x.x, ax.x), fmaxf(x.y, ax.y));
              else q = make_float2(fminf(x.x, ax.x), fminf(x.y, ax.y));
              accS[half * 2 + i2] = __fadd2_rn(accS[half * 2 + i2], q);
              accQ[half * 2 + i2] = __ffma2_rn(q, q, accQ[half * 2 + i2]);
              P[par][i2] = q;
            }
          }
#pragma unroll
          for (int i2 = 0; i2 < 2; ++i2) {
            pk[i2][gp * 2] = pack_half2(P[0][i2].x, P[1][i2].x);
            pk[i2][gp * 2 + 1] = pack_half2(P[0][i2].y, P[1][i2].y);
            if constexpr (NSPLIT == 2) {
              pl[i2][gp * 2] = pack_residual2(P[0][i2].x, P[1][i2].x, pk[i2][gp * 2]);
              pl[i2][gp * 2 + 1] = pack_residual2(P[0][i2].y, P[1][i2].y, pk[i2][gp * 2 + 1]);
            }
          }
        }
#pragma unroll
        for (int i2 = 0; i2 < 2; ++i2) {
          const int rl = (half * 2 + i2) * 32 + warp * 4 + rg;
          *reinterpret_cast<uint4*>(a_tile + sw128_offset(rl, c8)) = make_uint4(pk[i2][0], pk[i2][1], pk[i2][2], pk[i2][3]);
          if constexpr (NSPLIT == 2)
            *reinterpret_cast<uint4*>(a_tile + kAChunkBytes + sw128_offset(rl, c8)) = make_uint4(pl[i2][0], pl[i2][1], pl[i2][2], pl[i2][3]);
        }
      };
      Step sa, sb;
      issue(0, 0, sa);
#pragma unroll 1
      for (int j = 0; j < NCH; ++j) {
        const int s = j % kStages, u = j / kStages;
        issue(j, 1, sb);
        if (u > 0) mbar_wait(empty + s, (u - 1) & 1, 400 + j);
        compute(j, 0, sa);
        if (j + 1 < NCH) issue(j + 1, 0, sa);
        compute(j, 1, sb);
        fence_proxy_async();
        mbar_arrive(full_a + s);
      }
#pragma unroll
      for (int it = 0; it < 4; ++it) {
        if (rflag[it] & 1024) {
          const int sg = rflag[it] & 255;
          const float sv = accS[it].x + accS[it].y, qv = accQ[it].x + accQ[it].y;
          if (sg == 0) { qstat.s0 += sv; qstat.q0 += qv; }
          else if (sg == 1) { qstat.s1 += sv; qstat.q1 += qv; }
          else { atomicAdd(seg_acc + 2 * sg, sv); atomicAdd(seg_acc + 2 * sg + 1, qv); }
        }
      }
    } else
    for (int j = 0; j < NCH; ++j) {
      const int s = j % kStages, u = j / kStages;
      if (u > 0) mbar_wait(empty + s, (u - 1) & 1, 400 + j);
      uint8_t* a_tile = smem + s * STAGE;
      {  // MODE 2 (MODE 0 and 1 have their own software-pipelined loops above)
        const int kc = j * 64 + c8 * 8;
        const bool has_norm = p.norm.gamma != nullptr;
        float ga[8], be[8], go[8], bo[8];
        if (MODE == 2) {
          if (has_norm) {
#pragma unroll
            for (int i = 0; i < 8; ++i) { ga[i] = __ldg(p.norm.gamma + kc + i); be[i] = __ldg(p.norm.beta + kc + i); }
          }
#pragma unroll
          for (int i = 0; i < 8; ++i) { go[i] = __ldg(p.g_o + kc + i); bo[i] = __ldg(p.b_o + kc + i); }
        }
        float4 x0[4], x1[4];
#pragma unroll
        for (int it = 0; it < 4; ++it) {
          const int rl = it * 32 + warp * 4 + rg;
          if (rl < nrows) {
            const float4* src = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p.in) + (int64_t)(r0 + rl) * kC + kc);
            x0[it] = __ldg(src);
            x1[it] = __ldg(src + 1);
          } else {
            x0[it] = x1[it] = make_float4(0.f, 0.f, 0.f, 0.f);
          }
        }
#pragma unroll
        for (int it = 0; it < 4; ++it) {
          const int rl = it * 32 + warp * 4 + rg;
          float y[8] = {x0[it].x, x0[it].y, x0[it].z, x0[it].w, x1[it].x, x1[it].y, x1[it].z, x1[it].w};
          if (rl < nrows) {
            const int sg = smap.seg(r0 + rl);
            const float2 mr = tab_a[sg];
            if (MODE == 0) {
              // gamma / beta of the stream norm live in the weight image and the bias: A = (x - mean) * rstd
              const float nb = -mr.x * mr.y;
#pragma unroll
              for (int i = 0; i < 8; ++i) y[i] = fmaf(y[i], mr.y, nb);
            } else {
              if (has_norm) {
#pragma unroll
                for (int i = 0; i < 8; ++i) y[i] = ((y[i] - mr.x) * mr.y) * ga[i] + be[i];
              }
              const float2 mo = tab_b[sg];
#pragma unroll
              for (int i = 0; i < 8; ++i) y[i] = ((prelu(y[i], p.slope_o) - mo.x) * mo.y) * go[i] + bo[i];
            }
          }
          const uint4 pk = make_uint4(pack_half2(y[0], y[1]), pack_half2(y[2], y[3]), pack_half2(y[4], y[5]),
                                      pack_half2(y[6], y[7]));
          *reinterpret_cast<uint4*>(a_tile + sw128_offset(rl, c8)) = pk;
          if (NSPLIT == 2) {
            float r[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) r[i] = y[i] - __half2float(__float2half_rn(y[i]));   // exact residual in fp32
            const uint4 pl = make_uint4(pack_half2(r[0], r[1]), pack_half2(r[2], r[3]), pack_half2(r[4], r[5]),
                                        pack_half2(r[6], r[7]));
            *reinterpret_cast<uint4*>(a_tile + kAChunkBytes + sw128_offset(rl, c8)) = pl;
          }
        }
      }
      fence_proxy_async();
      mbar_arrive(full_a + s);
    }
    if (MODE == 1) qstat.flush_warp(slots, warp);

    // ------------------------------------------------------------ epilogue (warps 0-7)
    // warp w reads TMEM lanes 32*(w%4).. (rows) and columns (w/4)*NT/2 .. in chunks of 32.
    mbar_wait(acc_full, 0, 500);
    tc_fence_after();
    const int lq = warp & 3, ch = warp >> 2;
    float* stg = reinterpret_cast<float*>(smem) + warp * (32 * kStgPitch);  // aliases the (now idle) stage buffers
    const int my_rl = lq * 32 + lane;       // the row this thread owns in TMEM
    float2 rowacc2 = make_float2(0.f, 0.f);
    SegStat2 ostat;
    constexpr int NCC = NT / 64;            // 32-column chunks per column half
    if constexpr (MODE == 0 && H16) {
      // conv1: the thread that owns TMEM lane (= row) my_rl finishes its 32 columns itself - bias, PReLU, statistics,
      // fp16 pack - and parks them in a row-major tile in shared memory (pitch 528 B: conflict-free 16 B stores);
      // when both column halves are in, one TMA bulk store per row (512 contiguous bytes) writes the tile. No fp32
      // transpose through shared memory, no per-element segment routing (a row has ONE segment), no store instructions
      // in the warps: the staged version spent half the CTA's lifetime in its copy-out (12 k of 24 k cycles).
      constexpr int kRowPitch = kC * 2 + 16;
      uint8_t* tile = smem;                                   // aliases the (now idle) stage buffers: 128 x 528 B
      const bool valid = my_rl < nrows;
      const float2 sl2 = make_float2(p.slope, p.slope);
      float2 s2 = make_float2(0.f, 0.f), q2 = make_float2(0.f, 0.f);
      for (int cc = 0; cc < NCC; ++cc) {
        const int col0 = ch * (NT / 2) + cc * 32;
        float v[32];
        tmem_ld32(tmem_base + ((uint32_t)(lq * 32) << 16) + (uint32_t)col0, v);
        uint4* dst = reinterpret_cast<uint4*>(tile + my_rl * kRowPitch + col0 * 2);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          uint32_t h[4];
#pragma unroll
          for (int k = 0; k < 2; ++k) {
            const int c = 8 * i + 4 * k;
            const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.bias + col0 + c));   // same address in every lane
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
          dst[i] = make_uint4(h[0], h[1], h[2], h[3]);
        }
      }
      if (valid) {
        const int sg = smap.seg(r0 + my_rl);
        const float sv = s2.x + s2.y, qv = q2.x + q2.y;
        if (sg == 0) { ostat.s0 = sv; ostat.q0 = qv; }
        else if (sg == 1) { ostat.s1 = sv; ostat.q1 = qv; }
        else { atomicAdd(seg_acc + 2 * sg, sv); atomicAdd(seg_acc + 2 * sg + 1, qv); }
      }
      fence_proxy_async();                                     // our generic-proxy stores -> visible to the bulk copy
      asm volatile("bar.sync 1, 256;" ::: "memory");          // both column halves of every row are in the tile
      if (ch == 0 && valid) {
        bulk_copy_s2g(reinterpret_cast<__half*>(p.out) + (int64_t)(r0 + my_rl) * p.out_stride, tile + my_rl * kRowPitch, kC * 2);
        bulk_commit_group();
        bulk_wait_read_all();                                  // the tile must outlive the copy's reads
      }
    } else
    for (int cc = 0; cc < NCC; ++cc) {
      const int col0 = ch * (NT / 2) + cc * 32;
      float v[32];
      tmem_ld32(tmem_base + ((uint32_t)(lq * 32) << 16) + (uint32_t)col0, v);
      if (MODE == 1) {
#pragma unroll
        for (int i = 0; i < 16; ++i) rowacc2 = __fadd2_rn(rowacc2, make_float2(v[2 * i], v[2 * i + 1]));
      }
      __syncwarp();
#pragma unroll
      for (int i = 0; i < 8; ++i)
        *reinterpret_cast<float4*>(stg + lane * kStgPitch + i * 4) = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
      __syncwarp();
      // coalesced copy-out: 8 lanes x float4 = one 128 B row segment, 4 rows per instruction
      const int c4 = (lane & 7) * 4;
      const int gcol = (MODE == 2 ? by * NT : 0) + col0 + c4;
      float4 bias4 = make_float4(0.f, 0.f, 0.f, 0.f);
      if (MODE != 1) bias4 = __ldg(reinterpret_cast<const float4*>(p.bias + gcol));
      float4 cs0 = make_float4(0.f, 0.f, 0.f, 0.f), cs1 = cs0;   // column sums of the tile's 1st / 2nd utterance
      // FAST: a full tile that touches at most two utterances (every tile but the tensor's last when T >= 128): no
      // per-row bounds test and a two-way segment select, so the eight unrolled rows are straight-line code the
      // scheduler can interleave; the guarded variant wrapped every row in its own divergence region, which serialised
      // them (2000-2900 cycles per 32-column chunk in the clock64 timeline).
      auto copy_out = [&](auto fast_tag) {
      constexpr bool FAST = decltype(fast_tag)::value;
#pragma unroll
      for (int it = 0; it < 8; ++it) {
        const int i = it * 4 + (lane >> 3);
        const int rl = lq * 32 + i;
        if (FAST || rl < nrows) {
          float4 o = *reinterpret_cast<const float4*>(stg + i * kStgPitch + c4);
          const int row = r0 + rl;
          const int sg = FAST ? (row >= smap.e1 ? 1 : 0) : smap.seg(row);
          if (MODE == 0) {
            // bias + PReLU (max(x, a x) for a <= 1, min otherwise: AMAX) + statistics on the packed fp32 pipe
            const float2 sl2 = make_float2(p.slope, p.slope);
            const float2 x0 = __fadd2_rn(make_float2(o.x, o.y), make_float2(bias4.x, bias4.y));
            const float2 x1 = __fadd2_rn(make_float2(o.z, o.w), make_float2(bias4.z, bias4.w));
            const float2 a0 = __fmul2_rn(sl2, x0), a1 = __fmul2_rn(sl2, x1);
            if constexpr (AMAX) o = make_float4(fmaxf(x0.x, a0.x), fmaxf(x0.y, a0.y), fmaxf(x1.x, a1.x), fmaxf(x1.y, a1.y));
            else o = make_float4(fminf(x0.x, a0.x), fminf(x0.y, a0.y), fminf(x1.x, a1.x), fminf(x1.y, a1.y));
            const float2 r0 = make_float2(o.x, o.y), r1 = make_float2(o.z, o.w);
            const float2 sv = __fadd2_rn(r0, r1), qv = __ffma2_rn(r1, r1, __fmul2_rn(r0, r0));
            const float s = sv.x + sv.y, q = qv.x + qv.y;
            if (sg == 0) { ostat.s0 += s; ostat.q0 += q; }
            else if (FAST || sg == 1) { ostat.s1 += s; ostat.q1 += q; }
            else { atomicAdd(seg_acc + 2 * sg, s); atomicAdd(seg_acc + 2 * sg + 1, q); }
          } else if (MODE == 2) {
            o.x += bias4.x; o.y += bias4.y; o.z += bias4.z; o.w += bias4.w;
          } else {
            if (sg == 0) {
              const float2 a = __fadd2_rn(make_float2(cs0.x, cs0.y), make_float2(o.x, o.y)), b2 = __fadd2_rn(make_float2(cs0.z, cs0.w), make_float2(o.z, o.w));
              cs0 = make_float4(a.x, a.y, b2.x, b2.y);
            } else if (FAST || sg == 1) {
              const float2 a = __fadd2_rn(make_float2(cs1.x, cs1.y), make_float2(o.x, o.y)), b2 = __fadd2_rn(make_float2(cs1.z, cs1.w), make_float2(o.z, o.w));
              cs1 = make_float4(a.x, a.y, b2.x, b2.y);
            }
            else {  // only when T < 128
              double* dst = p.colsum + (size_t)(b_first + sg) * kC + col0 + c4;
              atomicAdd(dst, (double)o.x); atomicAdd(dst + 1, (double)o.y);
              atomicAdd(dst + 2, (double)o.z); atomicAdd(dst + 3, (double)o.w);
            }
          }
          if (H16 && MODE != 2)
            *reinterpret_cast<uint2*>(reinterpret_cast<__half*>(p.out) + (int64_t)row * p.out_stride + gcol) =
                make_uint2(pack_half2(o.x, o.y), pack_half2(o.z, o.w));
          else
            *reinterpret_cast<float4*>(reinterpret_cast<float*>(p.out) + (int64_t)row * p.out_stride + gcol) = o;
        }
      }
      };
      if (nrows == kTileM && nseg <= 2) copy_out(std::true_type{}); else copy_out(std::false_type{});
      if (MODE == 1) {
        // column sums: fold the 4 row groups of the warp, then one global atomic per column and utterance
#pragma unroll
        for (int o = 8; o <= 16; o <<= 1) {
          cs0.x += __shfl_xor_sync(0xffffffffu, cs0.x, o); cs0.y += __shfl_xor_sync(0xffffffffu, cs0.y, o);
          cs0.z += __shfl_xor_sync(0xffffffffu, cs0.z, o); cs0.w += __shfl_xor_sync(0xffffffffu, cs0.w, o);
          cs1.x += __shfl_xor_sync(0xffffffffu, cs1.x, o); cs1.y += __shfl_xor_sync(0xffffffffu, cs1.y, o);
          cs1.z += __shfl_xor_sync(0xffffffffu, cs1.z, o); cs1.w += __shfl_xor_sync(0xffffffffu, cs1.w, o);
        }
        if (lane < 8) {
          double* dst = p.colsum + (size_t)b_first * kC + col0 + c4;
          atomicAdd(dst, (double)cs0.x); atomicAdd(dst + 1, (double)cs0.y);
          atomicAdd(dst + 2, (double)cs0.z); atomicAdd(dst + 3, (double)cs0.w);
          if (nseg > 1) {
            dst += kC;
            atomicAdd(dst, (double)cs1.x); atomicAdd(dst + 1, (double)cs1.y);
            atomicAdd(dst + 2, (double)cs1.z); atomicAdd(dst + 3, (double)cs1.w);
          }
        }
      }
    }
    if (MODE == 0) ostat.flush_warp(slots, warp);
    if (MODE == 1) {
      // row sums: the two column halves (warps w and w+4) own the same rows
      const float rowacc = rowacc2.x + rowacc2.y;
      if (ch == 1) rs_x[my_rl] = rowacc;
      asm volatile("bar.sync 1, 256;" ::: "memory");
      if (ch == 0 && my_rl < nrows) p.rowsum[r0 + my_rl] = rowacc + rs_x[my_rl];
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 9) tmem_dealloc(tmem_base, 256);
  Stat2* sdst = (MODE == 0) ? p.st_out : (MODE == 1 ? p.st_q : nullptr);
  if (sdst != nullptr && by == 0) seg_stats_commit(slots, 8, seg_acc, nseg, sdst + b_first);
}

template <int MODE, bool H16, bool AMAX = true, bool SPLIT = false>
void launch_mode(const TcParams& p, int ntiles_n, cudaStream_t st) {
  constexpr int NT = (MODE == 2) ? 192 : 256;
  constexpr int smem = kStages * ((MODE == 2 || SPLIT) ? 2 : 1) * (kAChunkBytes + NT * 128) + kAuxBytes + 1024 + (MODE == 1 ? kDconvWBytes : 0);
  dim3 grid((p.M + kTileM - 1) / kTileM, ntiles_n);
  if (MODE == 2) grid = dim3(grid.x * 3, 1);   // (ntiles_n == 3: decoded in the kernel)
  launch_k(k_tc_gemm<MODE, H16, AMAX, SPLIT>, grid, dim3(kThreads), smem, st, true, p);
}

}  // namespace

template <int MODE, bool H16, bool AMAX = true, bool SPLIT = false>
cudaError_t setup_one(int smem) {
  cudaFuncSetAttribute(k_tc_gemm<MODE, H16, AMAX, SPLIT>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  return cudaFuncSetAttribute(k_tc_gemm<MODE, H16, AMAX, SPLIT>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
}

cudaError_t tc_gemm_setup() {
  // two CTAs per SM need (almost) the whole shared-memory carveout
  const int s0 = kStages * (kAChunkBytes + 256 * 128) + kAuxBytes + 1024;
  const int s2 = kStages * 2 * (kAChunkBytes + 192 * 128) + kAuxBytes + 1024;
  cudaError_t e;
  if ((e = setup_one<0, false>(s0)) != cudaSuccess) return e;
  if ((e = setup_one<0, true>(s0)) != cudaSuccess) return e;
  if ((e = setup_one<0, false, false>(s0)) != cudaSuccess) return e;
  if ((e = setup_one<0, true, false>(s0)) != cudaSuccess) return e;
  if ((e = setup_one<1, false>(s0 + kDconvWBytes)) != cudaSuccess) return e;
  if ((e = setup_one<1, true>(s0 + kDconvWBytes)) != cudaSuccess) return e;
  if ((e = setup_one<1, false, false>(s0 + kDconvWBytes)) != cudaSuccess) return e;
  if ((e = setup_one<1, true, false>(s0 + kDconvWBytes)) != cudaSuccess) return e;
  // split-precision ("accurate") variants: fp32 activations, [A_hi][A_lo][W_hi][W_lo] stages
  const int s0s = kStages * 2 * (kAChunkBytes + 256 * 128) + kAuxBytes + 1024;
  if ((e = setup_one<0, false, true, true>(s0s)) != cudaSuccess) return e;
  if ((e = setup_one<0, false, false, true>(s0s)) != cudaSuccess) return e;
  if ((e = setup_one<1, false, true, true>(s0s + kDconvWBytes)) != cudaSuccess) return e;
  if ((e = setup_one<1, false, false, true>(s0s + kDconvWBytes)) != cudaSuccess) return e;
  return setup_one<2, false>(s2);
}

void launch_tc_conv1(const Conv1Params& c, cudaStream_t st) {
  TcParams p{};
  p.M = c.M; p.T = c.T; p.B = c.B;
  p.w_img = c.w_img; p.w_img_lo = c.w_img_lo; p.in = c.w_in; p.norm = c.norm;
  p.bias = c.bias_f; p.slope = c.slope;
  p.out = c.p_out; p.out_stride = kC; p.st_out = c.st_p;
  if (c.split) {   // split-precision operands, fp32 p
    if (c.slope <= 1.f) launch_mode<0, false, true, true>(p, 1, st); else launch_mode<0, false, false, true>(p, 1, st);
  } else if (c.slope <= 1.f) {
    if (c.half_io) launch_mode<0, true, true>(p, 1, st); else launch_mode<0, false, true>(p, 1, st);
  } else {
    if (c.half_io) launch_mode<0, true, false>(p, 1, st); else launch_mode<0, false, false>(p, 1, st);
  }
}

void launch_tc_dconv(const DconvParams& c, cudaStream_t st) {
  TcParams p{};
  p.M = c.M; p.T = c.T; p.B = c.B;
  p.w_img = c.w_img; p.w_img_lo = c.w_img_lo; p.in = c.p_in;
  p.st_p = c.st_p; p.wtab = c.wtab; p.bog = c.bog;
  p.slope2 = c.slope2; p.dil = c.dil; p.st_q = c.st_q;
  p.out = c.racc; p.out_stride = kC; p.rowsum = c.rowsum; p.colsum = c.colsum;
  if (c.split) {   // split-precision operands, fp32 p and racc
    if (c.slope2 <= 1.f) launch_mode<1, false, true, true>(p, 1, st); else launch_mode<1, false, false, true>(p, 1, st);
  } else if (c.slope2 <= 1.f) {
    if (c.half_io) launch_mode<1, true, true>(p, 1, st); else launch_mode<1, false, true>(p, 1, st);
  } else {
    if (c.half_io) launch_mode<1, true, false>(p, 1, st); else launch_mode<1, false, false>(p, 1, st);
  }
}

void launch_tc_outconv(const OutConvParams& c, cudaStream_t st) {
  TcParams p{};
  p.M = c.M; p.T = c.T; p.B = c.B;
  p.w_img = c.w_img; p.w_img_lo = c.w_img_lo; p.in = c.w_in; p.norm = c.norm;
  p.slope_o = c.slope_o; p.st_o = c.st_o; p.g_o = c.g_o; p.b_o = c.b_o;
  p.bias = c.bias;
  p.out = c.logits; p.out_stride = kLogitStride;
  launch_mode<2, false>(p, 3, st);
}

}  // namespace septfa
