// Back-end kernels: VAD head (+ threshold / [1,0,1] smoothing), and mask application fused with the
// inverse STFT overlap-add and the optional torch-layout exports.
// Reference: model/model.py:173-179 (VAD), :423-457 (masks, noisy phase, inference gating),
// :460 (InverseSpectrogram -> torch.istft).
#include "kernels.h"
#include "fft512.cuh"
#include "tc_common.cuh"

namespace septfa {

// ------------------------------------------------------------------------------------------
// VAD head. VAD.common.conv1_1 (257 -> 4, k5, pad 2) is linear in the logits, so its per-frame partial products
//   part[row][s][k*4+j] = sum_f w[j][f][k] * logit[row][s*257 + f]
// are produced by the output convolution itself as 40 extra columns (composite weights, septfa_abi.cu) in the padding
// of the logits rows; this kernel combines the taps.
// Tap combination + PReLU + GroupNorm(1,4) over the [4,T] plane -> output_layer_vad (4 -> 1, k3, pad 1)
// -> sigmoid; then the inference-only threshold (>=) and [1,0,1] neighbour-OR smoothing with edge copy
// (model.py:173-179, 449-451). One CTA owns one (utterance, speaker): its statistics need no atomics.
__global__ void __launch_bounds__(256) k_vad_final(VadParams p) {
  __shared__ double red[2][8];
  __shared__ float2 s_mr;
  pdl_launch_dependents();
  pdl_wait();
  const int bs = blockIdx.x, b = bs >> 1, s = bs & 1;
  float* c4 = p.c4 + (int64_t)bs * p.T * 4;
  float* prob = p.prob + (int64_t)bs * p.T;
  double sum = 0.0, sumsq = 0.0;
  for (int t = threadIdx.x; t < p.T; t += blockDim.x) {
    float c[4] = {p.b1[0], p.b1[1], p.b1[2], p.b1[3]};
#pragma unroll
    for (int k = 0; k < 5; ++k) {
      const int tt = t + k - 2;
      if (tt < 0 || tt >= p.T) continue;
      const float4 v = __ldg(reinterpret_cast<const float4*>(p.logits + ((int64_t)b * p.T + tt) * kLogitStride + kVadCol0 + s * 20 + k * 4));
      c[0] += v.x; c[1] += v.y; c[2] += v.z; c[3] += v.w;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      c[j] = prelu(c[j], p.slope);
      sum += c[j];
      sumsq += (double)c[j] * c[j];
    }
    *reinterpret_cast<float4*>(c4 + (int64_t)t * 4) = make_float4(c[0], c[1], c[2], c[3]);
  }
  sum = warp_sum(sum);
  sumsq = warp_sum(sumsq);
  if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = sum; red[1][threadIdx.x >> 5] = sumsq; }
  __syncthreads();
  if (threadIdx.x == 0) {
    Stat2 st{0.0, 0.0};
    for (int i = 0; i < 8; ++i) { st.s += red[0][i]; st.ss += red[1][i]; }
    s_mr = stat_mean_rstd(&st, 1.0 / (4.0 * p.T), 1e-8f);
  }
  __syncthreads();
  const float2 mr = s_mr;
  for (int t = threadIdx.x; t < p.T; t += blockDim.x) {
    float acc = p.b2;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const int tt = t + k - 1;
      if (tt < 0 || tt >= p.T) continue;
      const float4 c = *reinterpret_cast<const float4*>(c4 + (int64_t)tt * 4);  // written by this CTA above
      acc += p.w2[0 * 3 + k] * (((c.x - mr.x) * mr.y) * p.g[0] + p.be[0]);
      acc += p.w2[1 * 3 + k] * (((c.y - mr.x) * mr.y) * p.g[1] + p.be[1]);
      acc += p.w2[2 * 3 + k] * (((c.z - mr.x) * mr.y) * p.g[2] + p.be[2]);
      acc += p.w2[3 * 3 + k] * (((c.w - mr.x) * mr.y) * p.g[3] + p.be[3]);
    }
    prob[t] = sigmoidf_acc(acc);
  }
  if (!p.do_smooth) return;
  __syncthreads();  // prob[] written by this CTA is visible to it after the barrier
  float* sm = p.smooth + (int64_t)bs * p.T;
  for (int t = threadIdx.x; t < p.T; t += blockDim.x) {
    const float d = prob[t] >= p.thr ? 1.f : 0.f;
    float v = d;
    if (t > 0 && t < p.T - 1) {
      const float dl = prob[t - 1] >= p.thr ? 1.f : 0.f;
      const float dr = prob[t + 1] >= p.thr ? 1.f : 0.f;
      v = fminf(dl + dr, 1.f);
    }
    sm[t] = v;
  }
}

void launch_vad(const VadParams& p, cudaStream_t st) {
  launch_k(k_vad_final, dim3(p.B * 2), dim3(256), 0, st, true, p);
}

// ------------------------------------------------------------------------------------------
// Mask application + inverse STFT + overlap-add, and the optional torch-layout exports, from one read of S and the logits.
// One CTA = 15 consecutive 256-sample output blocks of one utterance, BOTH speakers: the two Hermitian spectra share one
// complex FFT (Z = E0 + i E1 -> z = e0 + i e1). The 16 frames the blocks need are transformed four at a time by the CTA's
// four 64-thread groups (radix-8 FFT, fft512.cuh).
//   E_s[f] = S[t,f] * sigmoid(logit[s,f,t]) * gate[s,t]                    (model.py:429-437,452-455)
//   out[256 j + n] = (w[256+n] fr_j[256+n] + w[n] fr_{j+1}[n]) / (w[256+n]^2 + w[n]^2)        (:460)
// The CTA's rows of S and of the logits are staged in shared memory by bulk copies issued at the start, one mbarrier per
// round of 4 frames, so round 0 waits only for its own rows and the later rounds' rows arrive during its FFT. After the
// last round the same staged rows feed the exports (est, mask, logits in the reference's [.., 257, T] layouts, T
// contiguous) of the CTA's 15 owned frames j0 .. j0 + 14; the 16th frame belongs to the next CTA.
constexpr int kIstftBlocks = 15;   // output blocks per CTA = 16 frames in 4 rounds of 4 FFTs (one frame of overlap with the neighbour CTA: 6 % redundant)
constexpr int kIstftFrames = kIstftBlocks + 1;
constexpr int kIstftRounds = kIstftFrames / 4;
// A round's 4 rows of S are contiguous in the workspace (8224 B), but a row starts 16-byte aligned only at even row
// indices: the copy takes the 16-byte-aligned superset. It ends inside S's allocation, whose size is rounded up to 256 B.
constexpr int kStageSBytes = 4 * kBins * (int)sizeof(float2) + 16;
constexpr int kStageLgCols = 516;  // logits columns 0..515 (2064 B, a multiple of 16); the VAD partials from kVadCol0 on stay behind

// Without exports (the lean path): the same mask / iSTFT / overlap-add with the next round's operands prefetched into
// registers instead of staged in shared memory - 3 CTAs per SM instead of 2, measured slightly faster end to end.
__global__ void __launch_bounds__(256, 3) k_mask_istft(const float2* __restrict__ S, const float* __restrict__ logits,
                                                    const float* __restrict__ gate, const float* __restrict__ window,
                                                    const float2* __restrict__ twiddle, int64_t L, int T,
                                                    float* __restrict__ out) {
  __shared__ float2 buf[4][kFftPad];
  __shared__ float2 tw[kNfft];
  __shared__ float2 carry[kHop];  // windowed second half of the last frame of the previous round
  const int tid = threadIdx.x, grp = tid >> 6, j = tid & 63, b = blockIdx.y;
  const int j0 = blockIdx.x * kIstftBlocks;
  tw[tid] = __ldg(twiddle + tid);
  tw[tid + 256] = __ldg(twiddle + tid + 256);
  const float w_lo = __ldg(window + tid), w_hi = __ldg(window + kHop + tid);
  const float sc = 1.f / (float)kNfft;
  const float inv_env = 1.f / (w_hi * w_hi + w_lo * w_lo), inv_env_tail = 1.f / (w_hi * w_hi);   // one division per thread, not per sample
  pdl_launch_dependents();
  pdl_wait();
  float* out0 = out + ((int64_t)b * 2) * L;
  float* out1 = out0 + L;
  const int t_last = min(j0 + kIstftBlocks, T - 1);   // frames j0 .. t_last
  // A frame's operands (its row of S, its two rows of mask logits, its gates) are fetched one round AHEAD into registers:
  // the loads of round r + 1 are in flight during the FFT and the overlap-add of round r. Without that every round began
  // with a full HBM latency that only the other CTAs of the SM could cover (issue-active 36 %).
  struct FrameOps { float2 sv[4]; float l0[4], l1[4]; float g0, g1; };
  auto fetch = [&](int round, FrameOps& fo) {
    const int t = j0 + round * 4 + grp;
    if (t <= t_last) {
      const int64_t row = (int64_t)b * T + t;
      fo.g0 = fo.g1 = 1.f;
      if (gate != nullptr) {
        fo.g0 = __ldg(gate + ((int64_t)b * 2) * T + t);
        fo.g1 = __ldg(gate + ((int64_t)b * 2 + 1) * T + t);
      }
      const float* lr = logits + row * kLogitStride;
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int f = j + 64 * r, ff = f >= 1 ? f : 256;   // the thread of bin 0 (DC: zero) takes the Nyquist bin
        fo.sv[r] = __ldg(S + row * kBins + ff);
        fo.l0[r] = __ldg(lr + ff);
        fo.l1[r] = __ldg(lr + kBins + ff);
      }
    }
  };
  FrameOps fa, fb;
  fetch(0, fa);
#pragma unroll
  for (int round = 0; round < (kIstftBlocks + 1) / 4; ++round) {
    const int tbase = j0 + round * 4;
    if (tbase > t_last) break;                        // uniform
    const int t = tbase + grp;                        // this group's frame
    const bool vt = t <= t_last;
    FrameOps& cur = (round & 1) ? fb : fa;
    __syncthreads();                                  // previous round's reads of buf are done
    if (round + 1 < (kIstftBlocks + 1) / 4) fetch(round + 1, (round & 1) ? fa : fb);
    if (vt) {
      float2* bg = buf[grp];
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int f = j + 64 * r;  // 0..255
        const float2 sv = cur.sv[r];
        const float m0 = sigmoidf_fast(cur.l0[r]) * cur.g0, m1 = sigmoidf_fast(cur.l1[r]) * cur.g1;
        if (f >= 1) {
          const float a0 = sv.x * m0, b0 = sv.y * m0, a1 = sv.x * m1, b1 = sv.y * m1;
          bg[fft_idx(f)] = make_float2(a0 - b1, b0 + a1);               // E0[f] + i E1[f]
          bg[fft_idx(kNfft - f)] = make_float2(a0 + b1, a1 - b0);       // conj(E0[f]) + i conj(E1[f])
        } else {
          bg[fft_idx(0)] = make_float2(0.f, 0.f);                       // DC bin is zero
          bg[fft_idx(256)] = make_float2(sv.x * m0, sv.x * m1);         // irfft ignores the imaginary part of Nyquist
        }
      }
    }
    fft512_r8<true>(buf[grp], tw, j, grp);
    // output blocks of this round: block t-1 = second half of frame t-1 + first half of frame t, thread = sample n
    const int n = tid;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int tq = tbase + q;                       // frame held by group q
      if (tq > t_last) break;
      const float2 lo = buf[q][fft_idx(n)];
      const float2 first = make_float2(lo.x * sc * w_lo, lo.y * sc * w_lo);
      if (tq > j0) {
        float2 prev;
        if (q == 0) {
          prev = carry[n];
        } else {
          const float2 hi = buf[q - 1][fft_idx(kHop + n)];
          prev = make_float2(hi.x * sc * w_hi, hi.y * sc * w_hi);
        }
        const int64_t o = (int64_t)(tq - 1) * kHop + n;
        if (o < L) {
          out0[o] = (prev.x + first.x) * inv_env;
          out1[o] = (prev.y + first.y) * inv_env;
        }
      }
    }
    // carry the last frame of this round; the very last frame of the utterance has no successor (ragged tail)
    const int ql = min(3, t_last - tbase);
    const float2 hi = buf[ql][fft_idx(kHop + n)];
    const float2 second = make_float2(hi.x * sc * w_hi, hi.y * sc * w_hi);
    if (tbase + ql == T - 1 && T - 1 < j0 + kIstftBlocks) {
      const int64_t o = (int64_t)(T - 1) * kHop + n;
      if (o < L) {
        out0[o] = second.x * inv_env_tail;
        out1[o] = second.y * inv_env_tail;
      }
    }
    carry[n] = second;   // read only by the same thread in the next round
  }
}

void launch_mask_istft(const float2* S, const float* logits, const float* gate, const float* window,
                       const float2* twiddle, int B, int64_t L, int T, float* out, cudaStream_t st) {
  dim3 grid((T + kIstftBlocks - 1) / kIstftBlocks, B);
  launch_k(k_mask_istft, grid, dim3(256), 0, st, true, S, logits, gate, window, twiddle, L, T, out);
}

struct BackendSmem {
  float2 buf[4][kFftPad];
  float2 tw[kNfft];
  float2 carry[kHop];                           // windowed second half of the last frame of the previous round
  float lg[kIstftFrames][kStageLgCols];         // staged logits rows, column n = s * 257 + f
  alignas(16) uint8_t s[kIstftRounds][kStageSBytes];   // staged rows of S, round r at s[r] + (S row's address & 15)
  float g[2][kIstftFrames];                     // gates of the staged frames (1 without a gate)
  uint64_t bar[kIstftRounds];
};
constexpr int kBackendSmemBytes = (int)sizeof(BackendSmem);   // ~89 KB: 2 CTAs per SM

__global__ void __launch_bounds__(256, 2) k_mask_istft_export(const float2* __restrict__ S, const float* __restrict__ logits,
                                                           const float* __restrict__ gate, const float* __restrict__ window,
                                                           const float2* __restrict__ twiddle, int64_t L, int T,
                                                           float* __restrict__ out, float2* __restrict__ est,
                                                           float* __restrict__ mask, float* __restrict__ logits_out) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  BackendSmem& sm = *reinterpret_cast<BackendSmem*>(smem_raw);
  const int tid = threadIdx.x, grp = tid >> 6, j = tid & 63, b = blockIdx.y;
  const int j0 = blockIdx.x * kIstftBlocks;
  const int t_last = min(j0 + kIstftBlocks, T - 1);   // frames j0 .. t_last
  if (tid == 0) {
#pragma unroll
    for (int r = 0; r < kIstftRounds; ++r) tc::mbar_init(&sm.bar[r], 1);
    tc::fence_mbar_init();
  }
  sm.tw[tid] = __ldg(twiddle + tid);
  sm.tw[tid + 256] = __ldg(twiddle + tid + 256);
  const float w_lo = __ldg(window + tid), w_hi = __ldg(window + kHop + tid);
  const float sc = 1.f / (float)kNfft;
  const float inv_env = 1.f / (w_hi * w_hi + w_lo * w_lo), inv_env_tail = 1.f / (w_hi * w_hi);   // one division per thread, not per sample
  pdl_launch_dependents();
  pdl_wait();
  const int64_t row0 = (int64_t)b * T + j0;
  const float2* s_row0 = S + row0 * kBins;
  const uint32_t s_off = (uint32_t)reinterpret_cast<uintptr_t>(s_row0) & 15u;   // the same for every round (4 rows = 8224 B)
  if (tid == 0) {
    for (int r = 0; r < kIstftRounds; ++r) {
      const int n = min(4, t_last - (j0 + 4 * r) + 1);
      if (n <= 0) break;
      const uintptr_t a = reinterpret_cast<uintptr_t>(s_row0 + (int64_t)4 * r * kBins);
      const uintptr_t a0 = a & ~(uintptr_t)15, a1 = (a + (uintptr_t)n * kBins * sizeof(float2) + 15) & ~(uintptr_t)15;
      tc::mbar_expect_tx(&sm.bar[r], (uint32_t)(a1 - a0) + (uint32_t)n * kStageLgCols * sizeof(float));
      tc::bulk_copy_g2s(sm.s[r], reinterpret_cast<const void*>(a0), (uint32_t)(a1 - a0), &sm.bar[r]);
      for (int i = 0; i < n; ++i)
        tc::bulk_copy_g2s(sm.lg[4 * r + i], logits + (row0 + 4 * r + i) * kLogitStride, kStageLgCols * sizeof(float), &sm.bar[r]);
    }
  }
  if (tid < 2 * kIstftFrames) {
    const int s = tid / kIstftFrames, i = tid % kIstftFrames;
    sm.g[s][i] = (gate != nullptr && j0 + i <= t_last) ? __ldg(gate + ((int64_t)b * 2 + s) * T + j0 + i) : 1.f;
  }
  float* out0 = out + ((int64_t)b * 2) * L;
  float* out1 = out0 + L;
#pragma unroll
  for (int round = 0; round < kIstftRounds; ++round) {
    const int tbase = j0 + round * 4;
    if (tbase > t_last) break;                        // uniform
    const int t = tbase + grp;                        // this group's frame
    const bool vt = t <= t_last;
    __syncthreads();                                  // previous round's reads of buf are done (round 0: barriers initialised, gates staged)
    tc::mbar_wait(&sm.bar[round], 0, 0);
    if (vt) {
      float2* bg = sm.buf[grp];
      const float2* srow = reinterpret_cast<const float2*>(sm.s[round] + s_off) + grp * kBins;
      const float* lr = sm.lg[round * 4 + grp];
      const float g0 = sm.g[0][round * 4 + grp], g1 = sm.g[1][round * 4 + grp];
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int f = j + 64 * r;  // 0..255
        const int ff = f >= 1 ? f : 256;                // the thread of bin 0 (DC: zero) takes the Nyquist bin
        const float2 sv = srow[ff];
        const float m0 = sigmoidf_fast(lr[ff]) * g0, m1 = sigmoidf_fast(lr[kBins + ff]) * g1;
        if (f >= 1) {
          const float a0 = sv.x * m0, b0 = sv.y * m0, a1 = sv.x * m1, b1 = sv.y * m1;
          bg[fft_idx(f)] = make_float2(a0 - b1, b0 + a1);               // E0[f] + i E1[f]
          bg[fft_idx(kNfft - f)] = make_float2(a0 + b1, a1 - b0);       // conj(E0[f]) + i conj(E1[f])
        } else {
          bg[fft_idx(0)] = make_float2(0.f, 0.f);                       // DC bin is zero
          bg[fft_idx(256)] = make_float2(sv.x * m0, sv.x * m1);         // irfft ignores the imaginary part of Nyquist
        }
      }
    }
    fft512_r8<true>(sm.buf[grp], sm.tw, j, grp);
    // output blocks of this round: block t-1 = second half of frame t-1 + first half of frame t, thread = sample n
    const int n = tid;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int tq = tbase + q;                       // frame held by group q
      if (tq > t_last) break;
      const float2 lo = sm.buf[q][fft_idx(n)];
      const float2 first = make_float2(lo.x * sc * w_lo, lo.y * sc * w_lo);
      if (tq > j0) {
        float2 prev;
        if (q == 0) {
          prev = sm.carry[n];
        } else {
          const float2 hi = sm.buf[q - 1][fft_idx(kHop + n)];
          prev = make_float2(hi.x * sc * w_hi, hi.y * sc * w_hi);
        }
        const int64_t o = (int64_t)(tq - 1) * kHop + n;
        if (o < L) {
          out0[o] = (prev.x + first.x) * inv_env;
          out1[o] = (prev.y + first.y) * inv_env;
        }
      }
    }
    // carry the last frame of this round; the very last frame of the utterance has no successor (ragged tail)
    const int ql = min(3, t_last - tbase);
    const float2 hi = sm.buf[ql][fft_idx(kHop + n)];
    const float2 second = make_float2(hi.x * sc * w_hi, hi.y * sc * w_hi);
    if (tbase + ql == T - 1 && T - 1 < j0 + kIstftBlocks) {
      const int64_t o = (int64_t)(T - 1) * kHop + n;
      if (o < L) {
        out0[o] = second.x * inv_env_tail;
        out1[o] = second.y * inv_env_tail;
      }
    }
    sm.carry[n] = second;   // read only by the same thread in the next round
  }
  // Exports of the owned frames from the staged rows (every round that holds one has been waited for above). A half-warp
  // writes the contiguous run along T of one (speaker, bin) pair: lane i = frame j0 + i. Per element as the reference
  // layout asks: mask = sigmoid(lg), logits_out = lg, est = S * mask * gate (left to right, as k_export computed it).
  const int nown = min(kIstftBlocks, T - j0);
  const int i = tid & 15;
  if (i >= nown) return;
  const float2* srow_i = reinterpret_cast<const float2*>(sm.s[i >> 2] + s_off) + (i & 3) * kBins;
  const int64_t o_b = (int64_t)b * 2 * kBins * T + j0 + i;
  for (int p = tid >> 4; p < 2 * kBins; p += 16) {   // p = s * 257 + f: the logits column and the export row
    const float lg = sm.lg[i][p];
    const float m = sigmoidf_fast(lg);
    const int64_t o = o_b + (int64_t)p * T;
    if (mask != nullptr) mask[o] = m;
    if (logits_out != nullptr) logits_out[o] = lg;
    if (est != nullptr) {
      const int s = p >= kBins ? 1 : 0;
      const float2 sv = srow_i[p - s * kBins];
      const float g = sm.g[s][i];
      est[o] = make_float2(sv.x * m * g, sv.y * m * g);
    }
  }
}

cudaError_t backend_setup() {
  return cudaFuncSetAttribute(k_mask_istft_export, cudaFuncAttributeMaxDynamicSharedMemorySize, kBackendSmemBytes);
}

void launch_mask_istft_export(const float2* S, const float* logits, const float* gate, const float* window,
                              const float2* twiddle, int B, int64_t L, int T, float* out, float2* est, float* mask,
                              float* logits_out, cudaStream_t st) {
  dim3 grid((T + kIstftBlocks - 1) / kIstftBlocks, B);
  launch_k(k_mask_istft_export, grid, dim3(256), kBackendSmemBytes, st, true, S, logits, gate, window, twiddle, L, T, out,
           est, mask, logits_out);
}

}  // namespace septfa
