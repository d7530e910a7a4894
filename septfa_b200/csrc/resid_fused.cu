// Cluster-resident post-block update: TF-attention gates + both GroupNorm residual steps of a TCN block in ONE
// kernel. A thread-block cluster owns one utterance at a time; the residual stream tile (fp32) and the raw res_out
// accumulators (fp16) are read from HBM once into shared memory, the statistics of v cross the cluster through
// distributed shared memory in a fixed order, the statistics of the new stream leave as one double atomic pair per CTA,
// and the new stream is written back once. Replaces k_tf_gate + k_resid<0> + k_resid<1> (which read the two tensors
// twice) whenever an utterance fits a cluster: <= 8 CTAs up to T = 1152 frames (18 s), 16 CTAs (non-portable cluster size) up to
// T = 2304 (36.9 s).
// Reference: model/model.py:197-208 (TF_Attention), :347-352 (post-block norms).
#include <cooperative_groups.h>
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include "kernels.h"
#include "tc_common.cuh"

namespace cg = cooperative_groups;

namespace septfa {

namespace {

// shared-memory bytes per frame: the stream row (fp32, or fp16 in the half-stream mode) + the fp16 accumulator row
__host__ __device__ constexpr int row_bytes(bool in_half) { return kC * (in_half ? 2 : 4) + kC * 2; }

__device__ __forceinline__ float tf_chain2(const float* m, int n, int j, const float* w1, float b1, const float* w2,
                                           float b2, float slope) {
  // u1 = conv(k3,p1,d1)(m); u2 = conv(k3,p2,d2)(u1); both zero-pad their own input (model.py:184-185,190-191)
  float u2 = b2;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const int i = j + 2 * (k - 1);
    if (i < 0 || i >= n) continue;
    float u1 = b1;
#pragma unroll
    for (int kk = 0; kk < 3; ++kk) {
      const int ii = i + kk - 1;
      if (ii >= 0 && ii < n) u1 += w1[kk] * m[ii];
    }
    u2 += w2[k] * u1;
  }
  return sigmoidf_acc(prelu(u2, slope));
}

struct FusedParams {
  const void* w_in;         // [M,256] residual stream before the block: fp32, or fp16 (IN_H)
  void* w_out;              // [M,256] residual stream after the block: fp32, or fp16 (OUT_H); may alias w_in (same type)
  const __half* racc;       // [M,256] raw res_out accumulators (fp16)
  StreamNorm norm;          // affine that turns w into y
  const Stat2* st_q;        // [B] statistics of q (GroupNorm reg2, folded into res_out)
  const float* s3; const float* c03;
  const float* rowsum;      // [M]
  const double* colsum;     // [B,256]
  TfParams tf;
  int T, B, Tc;             // Tc = frames per CTA
  int discard;              // drop the consumed racc lines from the L2
  double inv_T, inv_HT, inv_CT;   // 1 / T, 1 / (512 T), 1 / (256 T): computed on the host (a double division is a long software routine,
                                  // and every thread of every CTA ran one before its first gate stage, thread 0 one per utterance)
  int mode;                 // LnMode
  const float* g_a; const float* b_a;   // ln_first / ln_modules
  Stat2* st_w;              // [B] statistics of the new stream (recursive mode), accumulated into a zeroed slot
};

// ---------------------------------------------------------------------------------------------------------------
// Persistent variant for utterances of at most 8 CTAs x kMaxTc frames (T <= 576, 9.2 s; the 4 s clips of the headline
// workload run with 8 CTAs x 32 frames, two CTAs per SM). The grid is as many clusters as the device keeps resident;
// a cluster walks utterances b = cluster, cluster + n, ... . One thread brings the cluster's tile of the NEXT
// utterance into the other half of a shared-memory double buffer with two TMA bulk copies (the rows of a CTA are
// contiguous in HBM: 1 KB of stream + 512 B of accumulators per frame) while all threads take the current utterance
// through gates -> statistics of v -> cluster exchange -> new stream, so the memory system always has the next tile
// in flight and CTA launch / teardown happens once per SM, not once per tile.
// The statistics of v cross the cluster with one push-style exchange (every CTA stores its partial into every peer's
// shared memory, ONE cluster barrier, then only local reads); the statistics of the new stream go out as one double
// atomic pair per CTA. A thread owns 4 channels (two packed pairs: FFMA2) of every 8th frame of the CTA's tile.
constexpr int kPersistThreads = 256;
constexpr int kPersistWarps = kPersistThreads / 32;
constexpr int kRowGroups = kPersistThreads / 64;   // a thread owns 4 channels of every kRowGroups-th frame of the tile
constexpr int kMaxTc = 144;

// IN_H / OUT_H: the stream is read / written as fp16 (the half-stream mode of the forward: blocks 1 .. n-1 read fp16,
// blocks 0 .. n-2 write fp16; the statistics of the new stream are those of the ROUNDED values, which is what the
// consumers normalise).
template <bool IN_H, bool OUT_H>
__global__ void __launch_bounds__(kPersistThreads, 4) k_resid_persist(FusedParams p) {
  using namespace tc;
  constexpr int kInBytes = IN_H ? 2 : 4;
  constexpr int kRowBytes = row_bytes(IN_H);
  extern __shared__ __align__(16) uint8_t smem[];
  cg::cluster_group cluster = cg::this_cluster();
  const int CS = (int)cluster.num_blocks(), rank = (int)cluster.block_rank();
  const int cluster_id = blockIdx.x / CS, n_clusters = gridDim.x / CS;
  const int TC = p.Tc;
  const int t0 = rank * TC, nt = min(TC, p.T - t0);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int c0 = (tid & 63) * 4, rg = tid >> 6;

  __shared__ float mf_s[kC], mt_s[kMaxTc + 8];                              // channel / time means (scratch of the gate stages)
  __shared__ __align__(16) float gf_s[2][kC], rb_s[2][kC], gt_s[2][kMaxTc];   // [parity of the utterance]
  __shared__ float red_a[16], red_b[16], red_c[8];
  __shared__ __align__(16) double xch[2][32];   // [parity][rank < 16][2]: partial (sum, sum of squares) of v from the peers
  __shared__ float s_sc[8];
  __shared__ float s_nx[2][4];
  __shared__ __align__(8) uint64_t full;
  __shared__ __align__(8) uint64_t xbar[2];     // [parity]: the peers' partials of v have arrived (16 bytes each, st.async)

  if (tid == 0) {
    mbar_init(&full, 1);
    mbar_init(&xbar[0], 1);
    mbar_init(&xbar[1], 1);
    fence_mbar_init();
  }
  cluster.barrier_arrive();   // "this CTA runs": peers wait for it before they store into our shared memory
  pdl_launch_dependents();
  __syncthreads();
  pdl_wait();

  auto fetch = [&](int b) {   // one thread: two bulk copies onto the tile's mbarrier
    const int64_t row0 = (int64_t)b * p.T + t0;
    mbar_expect_tx(&full, (uint32_t)nt * kRowBytes);
    bulk_copy_g2s(smem, reinterpret_cast<const uint8_t*>(p.w_in) + row0 * kC * kInBytes, (uint32_t)nt * kC * kInBytes, &full);
    bulk_copy_g2s(smem + (size_t)TC * kC * kInBytes, p.racc + row0 * kC, (uint32_t)nt * kC * 2, &full);
  };
  if (tid == 0 && cluster_id < p.B) fetch(cluster_id);

  const bool has_norm = p.norm.gamma != nullptr;
  const bool recursive = p.mode == LN_RECURSIVE;
  const double inv_T = p.inv_T;
  // static per-channel operands, once per CTA
  const float c03v = __ldg(p.c03 + tid), s3v = __ldg(p.s3 + tid);
  float4 g4 = make_float4(1.f, 1.f, 1.f, 1.f), b4 = make_float4(0.f, 0.f, 0.f, 0.f);
  if (has_norm) { g4 = __ldg(reinterpret_cast<const float4*>(p.norm.gamma + c0)); b4 = __ldg(reinterpret_cast<const float4*>(p.norm.beta + c0)); }
  float4 ga4 = make_float4(1.f, 1.f, 1.f, 1.f), ba4 = make_float4(0.f, 0.f, 0.f, 0.f);
  if (p.mode != LN_NONE) { ga4 = __ldg(reinterpret_cast<const float4*>(p.g_a + c0)); ba4 = __ldg(reinterpret_cast<const float4*>(p.b_a + c0)); }

  // per-utterance small operands, fetched one utterance ahead. The four scalars every thread needs (rstd and mean of
  // q, mean and rstd of the incoming stream) involve double arithmetic: ONE thread computes them for the next utterance
  // and leaves them in shared memory (s_nx[parity]); 16 warps repeating that code was a third of the kernel's issue slots.
  double csv = 0.0;
  float rsv = 0.f;
  auto scalars_for = [&](int b, int par, int which) {   // two threads (of different warps): which = 0 the statistics of q, 1 those of the stream
    if (which == 0) {
      const Stat2 sq{__ldg(&p.st_q[b].s), __ldg(&p.st_q[b].ss)};
      const float2 mrq = stat_mean_rstd(&sq, p.inv_HT, 1e-8f);
      s_nx[par][0] = mrq.y; s_nx[par][1] = mrq.x;
    } else {
      float2 my = make_float2(0.f, 1.f);
      if (has_norm) {
        const Stat2 sy{__ldg(&p.norm.st[b].s), __ldg(&p.norm.st[b].ss)};
        my = stat_mean_rstd(&sy, p.norm.inv_n, p.norm.eps);
      }
      s_nx[par][2] = my.x; s_nx[par][3] = my.y;
    }
  };
  auto fetch_small = [&](int b) {
    csv = __ldg(p.colsum + b * kC + tid);
    if (tid < nt + 6) {
      const int t = t0 - 3 + tid;
      rsv = (t >= 0 && t < p.T) ? __ldg(p.rowsum + (int64_t)b * p.T + t) : 0.f;
    }
  };
  // Gates of one utterance (model.py:197-208) in three stages separated by block barriers: affine of r from the reg2
  // statistics and channel means -> frequency gate chain and time means -> time gate chain. Inside the loop the stages
  // of the NEXT utterance ride on the barriers the current one needs anyway (after the cluster exchange, after the
  // statistics broadcast, after the final reduction), so the gates cost no barrier and no exposed latency of their own.
  static_assert(kPersistThreads == kC, "gate stages: one thread per channel");
  auto gate_stage0 = [&](int par) {
    const float ra = s_nx[par][0];
    const float rbv = c03v - ra * s_nx[par][1] * s3v;
    rb_s[par][tid] = rbv;
    mf_s[tid] = ra * (float)(csv * inv_T) + rbv;
    const float s = warp_sum(rbv);
    if (lane == 0) red_c[warp] = s;
  };
  auto gate_stage1 = [&](int par) {
    gf_s[par][tid] = p.tf.enabled ? tf_chain2(mf_s, kC, tid, p.tf.wf1, p.tf.bf1, p.tf.wf2, p.tf.bf2, p.tf.af) : 1.f;
    if (tid < nt + 6) {
      float rbsum = 0.f;
#pragma unroll
      for (int k = 0; k < kPersistWarps; ++k) rbsum += red_c[k];
      const int t = t0 - 3 + tid;
      mt_s[tid] = (t >= 0 && t < p.T) ? s_nx[par][0] * (rsv / (float)kC) + rbsum / (float)kC : 0.f;
    }
  };
  auto gate_stage2 = [&](int par) {
    if (tid < nt)
      gt_s[par][tid] = p.tf.enabled ? tf_chain2(mt_s + 3 - t0, p.T, t0 + tid, p.tf.wt1, p.tf.bt1, p.tf.wt2, p.tf.bt2, p.tf.at) : 1.f;
  };
  if (cluster_id < p.B) {
    fetch_small(cluster_id);
    if (tid == kPersistThreads - 1) scalars_for(cluster_id, 0, 0);
    if (tid == kPersistThreads - 33) scalars_for(cluster_id, 0, 1);
    __syncthreads();
    gate_stage0(0);
    __syncthreads();
    gate_stage1(0);
    __syncthreads();
    gate_stage2(0);
  }
  __syncthreads();

  // fixed-order block reduction of two floats; the double totals are valid in every lane of warp 0
  auto block_total = [&](float s, float q, double& ts, double& tq) {
    s = warp_sum(s);
    q = warp_sum(q);
    if (lane == 0) { red_a[warp] = s; red_b[warp] = q; }
    __syncthreads();
    if (warp == 0) {
      ts = warp_sum(lane < kPersistWarps ? (double)red_a[lane] : 0.0);
      tq = warp_sum(lane < kPersistWarps ? (double)red_b[lane] : 0.0);
    }
  };

  bool peers_up = false;
  for (int b = cluster_id, it = 0; b < p.B; b += n_clusters, ++it) {
    const int buf = it & 1;
    const uint8_t* w_s = smem;                                                                 // [TC][256] stream rows (fp32 / fp16)
    const __half* r_s = reinterpret_cast<const __half*>(smem + (size_t)TC * kC * kInBytes);    // [TC][256] fp16 accumulators
    auto load_w4 = [&](int i) -> float4 {     // this thread's 4 channels of frame i
      if constexpr (IN_H) {
        const uint2 hw = *reinterpret_cast<const uint2*>(w_s + ((size_t)i * kC + c0) * 2);
        const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&hw.x)), b = __half22float2(*reinterpret_cast<const __half2*>(&hw.y));
        return make_float4(a.x, a.y, b.x, b.y);
      } else {
        return *reinterpret_cast<const float4*>(w_s + ((size_t)i * kC + c0) * 4);
      }
    };
    const int b_next = b + n_clusters;
    const bool has_next = b_next < p.B;
    if (has_next) {
      fetch_small(b_next);                    // consumed by the gate stages further down
      if (tid == kPersistThreads - 1) scalars_for(b_next, buf ^ 1, 0);
      if (tid == kPersistThreads - 33) scalars_for(b_next, buf ^ 1, 1);
    }
    const float ra = s_nx[buf][0], mean_y = s_nx[buf][2], rstd_y = s_nx[buf][3];
    const float* gt_cur = gt_s[buf];

    // ---- per-thread channel coefficients, as two packed pairs (channels c0,c0+1 | c0+2,c0+3): FFMA2 on sm_100
    float2 Ay[2], By[2], G1[2], G2[2];
    {
      const float4 gf4 = *reinterpret_cast<const float4*>(gf_s[buf] + c0), rb4 = *reinterpret_cast<const float4*>(rb_s[buf] + c0);
      const float2 rs2 = make_float2(rstd_y, rstd_y), nm2 = make_float2(-mean_y, -mean_y), ra2 = make_float2(ra, ra);
      Ay[0] = __fmul2_rn(rs2, make_float2(g4.x, g4.y));
      Ay[1] = __fmul2_rn(rs2, make_float2(g4.z, g4.w));
      By[0] = __ffma2_rn(nm2, Ay[0], make_float2(b4.x, b4.y));
      By[1] = __ffma2_rn(nm2, Ay[1], make_float2(b4.z, b4.w));
      G1[0] = __fmul2_rn(ra2, make_float2(gf4.x, gf4.y));
      G1[1] = __fmul2_rn(ra2, make_float2(gf4.z, gf4.w));
      G2[0] = __fmul2_rn(make_float2(rb4.x, rb4.y), make_float2(gf4.x, gf4.y));
      G2[1] = __fmul2_rn(make_float2(rb4.z, rb4.w), make_float2(gf4.z, gf4.w));
    }
    mbar_wait(&full, it & 1, 700);   // the tile has landed (every thread observes the barrier itself)
    if (p.discard) {
      // racc is read exactly once, by this CTA, and it is in shared memory now: its lines in the L2 are dead but dirty (the
      // dconv kernel wrote them) - dropped here they are neither written to DRAM nor in the residual stream's way
      const uint8_t* rg = reinterpret_cast<const uint8_t*>(p.racc + ((int64_t)b * p.T + t0) * kC);
      for (int l = tid; l < nt * 4; l += kPersistThreads) asm volatile("discard.global.L2 [%0], 128;" ::"l"(rg + (size_t)l * 128) : "memory");
    }

    // ---- statistics of v = y + gt (G1 r + G2)  (recursive)  |  gt (G1 r + G2)  (residual) over the whole utterance
    float2 mv = make_float2(0.f, 1.f);
    if (p.mode != LN_NONE) {
      float2 s2 = make_float2(0.f, 0.f), q2 = make_float2(0.f, 0.f);
      for (int i0 = rg; i0 < nt; i0 += 4 * kRowGroups)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int i = i0 + kRowGroups * j;
        if (i >= nt) break;
        const float g = gt_cur[i];
        const float2 gt2 = make_float2(g, g);
        const float4 wv = load_w4(i);
        const uint2 hv = *reinterpret_cast<const uint2*>(r_s + i * kC + c0);
        const float2 r0 = __half22float2(*reinterpret_cast<const __half2*>(&hv.x));
        const float2 r1 = __half22float2(*reinterpret_cast<const __half2*>(&hv.y));
        float2 v0 = __fmul2_rn(gt2, __ffma2_rn(r0, G1[0], G2[0])), v1 = __fmul2_rn(gt2, __ffma2_rn(r1, G1[1], G2[1]));
        if (recursive) {
          v0 = __fadd2_rn(v0, __ffma2_rn(make_float2(wv.x, wv.y), Ay[0], By[0]));
          v1 = __fadd2_rn(v1, __ffma2_rn(make_float2(wv.z, wv.w), Ay[1], By[1]));
        }
        s2 = __fadd2_rn(s2, __fadd2_rn(v0, v1));
        q2 = __ffma2_rn(v0, v0, q2);
        q2 = __ffma2_rn(v1, v1, q2);
      }
      double ts = 0.0, tq = 0.0;
      block_total(s2.x + s2.y, q2.x + q2.y, ts, tq);
      if (!peers_up) { cluster.barrier_wait(); peers_up = true; }   // every peer is running: its shared memory may be written
      // Push-style exchange without a cluster barrier: every CTA sends its 16-byte partial to every peer with st.async, which
      // counts the bytes on the RECEIVER's mbarrier; a CTA then waits for its own 8 x 16 bytes. (cluster.sync() is
      // arrive.release + wait: the release fence first drained the previous utterance's 32 KB of global stores - MEMBAR /
      // ERRBAR were 7 % of the kernel's stall samples - and every CTA then waited for the slowest peer's drain.) A peer can
      // be at most one utterance ahead (it needs OUR next partial to go further), so two buffers / barriers suffice.
      if (warp == 0) {
        if (lane == 0) mbar_expect_tx(&xbar[buf], (uint32_t)CS * 16u);
        if (lane < CS) {
          uint32_t rdst, rbar;
          asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(rdst) : "r"(smem_u32(&xch[buf][2 * rank])), "r"((uint32_t)lane));
          asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(rbar) : "r"(smem_u32(&xbar[buf])), "r"((uint32_t)lane));
          asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.b64 [%0], {%1, %2}, [%3];" ::"r"(rdst),
                       "l"(__double_as_longlong(ts)), "l"(__double_as_longlong(tq)), "r"(rbar)
                       : "memory");
        }
      }
      if (tid == 0) {
        mbar_wait(&xbar[buf], (it >> 1) & 1, 710);
        Stat2 tot{0.0, 0.0};
        for (int r = 0; r < CS; ++r) { tot.s += xch[buf][2 * r]; tot.ss += xch[buf][2 * r + 1]; }
        const float2 m = stat_mean_rstd(&tot, p.inv_CT, 1e-5f);
        s_sc[4] = m.x;
        s_sc[5] = m.y;
      }
    }
    if (has_next) gate_stage0(buf ^ 1);
    __syncthreads();
    if (p.mode != LN_NONE) mv = make_float2(s_sc[4], s_sc[5]);

    // ---- new stream o = y + Av v + Bv, folded into one affine per operand:
    //   o = P w + Q + gt (R1 r + R2),   P = k Ay, Q = k By + Bv, R1 = Av G1, R2 = Av G2,  k = 1 + Av (recursive) | 1
    float2 P[2], Q[2], R1[2], R2[2];
    {
      float2 Av[2] = {make_float2(1.f, 1.f), make_float2(1.f, 1.f)}, Bv[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
      if (p.mode != LN_NONE) {
        const float2 rs2 = make_float2(mv.y, mv.y), nm2 = make_float2(-mv.x, -mv.x);
        Av[0] = __fmul2_rn(rs2, make_float2(ga4.x, ga4.y));
        Av[1] = __fmul2_rn(rs2, make_float2(ga4.z, ga4.w));
        Bv[0] = __ffma2_rn(nm2, Av[0], make_float2(ba4.x, ba4.y));
        Bv[1] = __ffma2_rn(nm2, Av[1], make_float2(ba4.z, ba4.w));
      }
      const float2 one2 = make_float2(1.f, 1.f);
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        const float2 kk = recursive ? __fadd2_rn(one2, Av[k]) : one2;
        P[k] = __fmul2_rn(kk, Ay[k]);
        Q[k] = __ffma2_rn(kk, By[k], Bv[k]);
        R1[k] = __fmul2_rn(Av[k], G1[k]);
        R2[k] = __fmul2_rn(Av[k], G2[k]);
      }
    }
    float2 s2 = make_float2(0.f, 0.f), q2 = make_float2(0.f, 0.f);
    uint64_t keep_policy;   // the new stream is read twice more (conv1, then this kernel again): last in line for eviction
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(keep_policy));
    uint8_t* wout = reinterpret_cast<uint8_t*>(p.w_out) + (((int64_t)b * p.T + t0) * kC + c0) * (OUT_H ? 2 : 4);
    for (int i0 = rg; i0 < nt; i0 += 4 * kRowGroups)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int i = i0 + kRowGroups * j;
      if (i >= nt) break;
      const float g = gt_cur[i];
      const float2 gt2 = make_float2(g, g);
      const float4 wv = load_w4(i);
      const uint2 hv = *reinterpret_cast<const uint2*>(r_s + i * kC + c0);
      const float2 r0 = __half22float2(*reinterpret_cast<const __half2*>(&hv.x));
      const float2 r1 = __half22float2(*reinterpret_cast<const __half2*>(&hv.y));
      float2 o0 = __ffma2_rn(gt2, __ffma2_rn(r0, R1[0], R2[0]), __ffma2_rn(make_float2(wv.x, wv.y), P[0], Q[0]));
      float2 o1 = __ffma2_rn(gt2, __ffma2_rn(r1, R1[1], R2[1]), __ffma2_rn(make_float2(wv.z, wv.w), P[1], Q[1]));
      if constexpr (OUT_H) {
        const __half2 h0 = __floats2half2_rn(o0.x, o0.y), h1 = __floats2half2_rn(o1.x, o1.y);
        o0 = __half22float2(h0);
        o1 = __half22float2(h1);
        *reinterpret_cast<uint2*>(wout + (int64_t)i * kC * 2) =
            make_uint2(*reinterpret_cast<const uint32_t*>(&h0), *reinterpret_cast<const uint32_t*>(&h1));
      } else {
        asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1, %2, %3, %4}, %5;" ::"l"(wout + (int64_t)i * kC * 4), "f"(o0.x), "f"(o0.y), "f"(o1.x),
                     "f"(o1.y), "l"(keep_policy)
                     : "memory");
      }
      s2 = __fadd2_rn(s2, __fadd2_rn(o0, o1));
      q2 = __ffma2_rn(o0, o0, q2);
      q2 = __ffma2_rn(o1, o1, q2);
    }
    if (has_next) gate_stage1(buf ^ 1);
    {
      double ts = 0.0, tq = 0.0;
      block_total(s2.x + s2.y, q2.x + q2.y, ts, tq);   // its barrier also orders stage 1 before stage 2 ...
      if (tid == 0) {
        if (has_next) fetch(b_next);                  // ... and every thread's last read of the tile before this refill
        if (recursive) { atomicAdd(&p.st_w[b].s, ts); atomicAdd(&p.st_w[b].ss, tq); }
      }
    }
    if (has_next) gate_stage2(buf ^ 1);
    __syncthreads();   // every thread is done with this buffer and the scratch arrays: the next fetch may overwrite it
  }
  if (!peers_up) cluster.barrier_wait();
}

}  // namespace

int resid_fused_cluster_size(int T) {   // 0: the utterance does not fit one cluster (the forward uses the streaming kernels)
  if (T > 16 * kMaxTc) return 0;
  if (T > 8 * kMaxTc) return 16;          // 18 .. 36 s: clusters of 16 CTAs (non-portable size, allowed per kernel in setup)
  return std::min(8, (T + 31) / 32);
}

typedef void (*ResidKernel)(FusedParams);
static ResidKernel resid_kernel(int in_half, int out_half) {
  return in_half ? (out_half ? k_resid_persist<true, true> : k_resid_persist<true, false>)
                 : (out_half ? k_resid_persist<false, true> : k_resid_persist<false, false>);
}

cudaError_t resid_fused_setup() {
  int dev = 0, optin = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  for (int v = 0; v < 4; ++v) {
    cudaFuncAttributes fa{};
    cudaError_t e = cudaFuncGetAttributes(&fa, resid_kernel(v >> 1, v & 1));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(resid_kernel(v >> 1, v & 1), cudaFuncAttributeMaxDynamicSharedMemorySize, optin - (int)fa.sharedSizeBytes);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(resid_kernel(v >> 1, v & 1), cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}

// Clusters of the persistent kernel the device keeps resident at once (0: none, or the query failed).
int resid_fused_resident_clusters(bool in_half, bool out_half, int T) {
  const int cs = resid_fused_cluster_size(T);
  if (cs == 0) return 0;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(cs * 1024);
  cfg.blockDim = dim3(kPersistThreads);
  cfg.dynamicSmemBytes = (size_t)((T + cs - 1) / cs) * row_bytes(in_half);
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = cs; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  int n = 0;
  if (cudaOccupancyMaxActiveClusters(&n, resid_kernel(in_half, out_half), &cfg) != cudaSuccess) { cudaGetLastError(); n = 0; }
  return n;
}

// Programmatic early launch of the persistent cluster kernel: only safe because its predecessor (the dconv kernel)
// does not trigger its dependents, so they launch as its CTAs exit. With the usual trigger at kernel entry the
// persistent grid became resident while the dconv grid's second wave still needed the SM slots (5.86 vs 5.09 ms per
// step); with the late trigger the early launch hides the launch latency instead (3.75 -> 3.70 ms).
void launch_resid_fused(const ResidParams& rp, const GateParams& gp, int clusters, cudaStream_t st) {
  const int cs = resid_fused_cluster_size(rp.T);
  FusedParams p{};
  p.w_in = rp.w_half_in ? rp.w_half_in : static_cast<const void*>(rp.w);
  p.w_out = rp.w_half_out ? rp.w_half_out : static_cast<void*>(rp.w);
  p.racc = reinterpret_cast<const __half*>(rp.racc); p.norm = rp.norm;
  p.st_q = gp.st_q; p.s3 = gp.s3; p.c03 = gp.c03; p.rowsum = gp.rowsum; p.colsum = gp.colsum; p.tf = gp.tf;
  p.T = rp.T; p.B = rp.B; p.Tc = (rp.T + cs - 1) / cs; p.discard = rp.discard;
  p.inv_T = 1.0 / (double)rp.T; p.inv_HT = 1.0 / ((double)kH * rp.T); p.inv_CT = 1.0 / ((double)kC * rp.T);
  p.mode = rp.mode; p.g_a = rp.g_a; p.b_a = rp.b_a; p.st_w = rp.st_w;
  const bool in_half = rp.w_half_in != nullptr;
  const size_t smem = (size_t)p.Tc * row_bytes(in_half);
  launch_k(resid_kernel(in_half, rp.w_half_out != nullptr), Grid(dim3(std::min(clusters, rp.B) * cs), cs), dim3(kPersistThreads),
           smem, st, true, p);
}

}  // namespace septfa
