// Front-end kernel: STFT (frame, window, 512-point shared-memory FFT), power-dB, activity gate and
// the statistics of the TCN input norm, fused: the dB spectrogram never goes to HBM.
// Reference: model/model.py:408-419 (Spectrogram/InputSpec -> torch.stft, AmplitudeToDB,
// activity_input Conv2d 3x3 + PReLU) and :333 (TCN.LN statistics).
#include "kernels.h"
#include "fft512.cuh"

namespace septfa {

// Launch context of the calling thread: every C-ABI entry binds its handle's context (kernels.h), so the "pdl" option,
// the SM count and the launch counter are per handle, not process-wide.
namespace { LaunchCtx g_default_ctx; thread_local LaunchCtx* t_ctx = nullptr; }
LaunchCtx& ctx() { return t_ctx ? *t_ctx : g_default_ctx; }
void bind_ctx(LaunchCtx* c) { t_ctx = c; }

// Per-pass twiddle table of the radix-8 FFT (layout: fft512.cuh), computed in double on the host.
void make_twiddles(float2* h) {
  const double tau = -2.0 * 3.14159265358979323846;
  for (int j = 0; j < 512; ++j) h[j] = make_float2(0.f, 0.f);
  for (int r = 1; r < 8; ++r) {
    for (int k = 0; k < 8; ++k) h[(r - 1) * 8 + k] = make_float2((float)cos(tau * r * k / 64.0), (float)sin(tau * r * k / 64.0));
    for (int k = 0; k < 64; ++k) h[64 + (r - 1) * 64 + k] = make_float2((float)cos(tau * r * k / 512.0), (float)sin(tau * r * k / 512.0));
  }
}

constexpr int kFrontFrames = 14;              // frames produced per CTA
constexpr int kFrontRows = kFrontFrames + 2;  // + one halo frame each side for the 3x3 gate
constexpr int kPPitch = kBins + 3;            // dB row: [0] = bin -1 (zero pad), [1..257] = bins, [258] = bin 257 (zero pad)

struct GateK { float k[9]; float bias, slope; int enabled; };

// One CTA = 14 consecutive frames of one utterance (+1 halo frame each side). The 16 frames form 8 pairs; two real
// frames share one complex FFT (z = a + i b; A[k] = (Z[k] + conj Z[N-k]) / 2, B[k] = (Z[k] - conj Z[N-k]) / 2i), and
// the CTA's four 64-thread groups run four radix-8 FFTs side by side (two rounds).
// torch.stft(center=True, pad_mode='reflect', onesided), no normalisation, DC bin zeroed (model.py:24,410);
// P = 10 log10(max(|S|^2, 1e-10)); spectrum *= PReLU(Conv2d 3x3 (zero pad 1) over the (257, T) plane),
// rows 1..256 feed the TCN (model.py:411-421).
template <bool SPECTRUM>
__global__ void __launch_bounds__(256) k_frontend(const float* __restrict__ x, int64_t L, int T,
                                                  const float* __restrict__ window, const float2* __restrict__ twiddle,
                                                  GateK gk, float2* __restrict__ S, float* __restrict__ z0,
                                                  float* __restrict__ dc_gated, Stat2* __restrict__ st0,
                                                  float* __restrict__ spectrum /*[B,257,T] or null*/) {
  __shared__ float2 buf[4][kFftPad];
  __shared__ float2 tw[kNfft];
  __shared__ float win[kNfft];
  __shared__ float P[kFrontRows][kPPitch];
  __shared__ float red[64];
  __shared__ double nyq[4][2][2];   // [group][warp of the group][frame a / b]: Nyquist bins recomputed in double
  __shared__ int nyq_flag[4];
  pdl_launch_dependents();
  const int tid = threadIdx.x, grp = tid >> 6, j = tid & 63;
  const int b = blockIdx.y, t0 = blockIdx.x * kFrontFrames;
  const float* xb = x + (int64_t)b * L;
  tw[tid] = __ldg(twiddle + tid);
  tw[tid + 256] = __ldg(twiddle + tid + 256);
  win[tid] = __ldg(window + tid);
  win[tid + 256] = __ldg(window + tid + 256);
  for (int i = tid; i < kFrontRows * kPPitch; i += 256) (&P[0][0])[i] = 0.f;  // zero padding of the gate conv
  pdl_wait();  // S / z0 / statistics of the previous forward may still be in use by its last kernels
  __syncthreads();

  for (int round = 0; round < 2; ++round) {
    const int la = 2 * (round * 4 + grp);  // local row of frame a (rows 0 and 15 are halo rows)
    const int ta = t0 - 1 + la, tb = ta + 1;
    const bool va = ta >= 0 && ta < T, vb = tb >= 0 && tb < T;
    // sample index within the utterance in 32 bits (check_forward_args bounds L), reflect padding of 256 samples
    const int Li = (int)L, ia0 = ta * kHop + j - kNfft / 2;
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      const int n = j + 64 * r;
      float a = 0.f, c = 0.f;
      int i = ia0 + 64 * r;
      int ib = i + kHop;
      if (i < 0) i = -i;
      if (i >= Li) i = 2 * (Li - 1) - i;
      if (ib < 0) ib = -ib;
      if (ib >= Li) ib = 2 * (Li - 1) - ib;
      const float w = win[n];
      if (va) a = __ldg(xb + i) * w;
      if (vb) c = __ldg(xb + ib) * w;
      buf[grp][fft_idx(n)] = make_float2(a, c);
    }
    fft512_r8<false>(buf[grp], tw, j, grp);
    // The Nyquist bin is REAL, X[256] = sum_n (-1)^n x[n] w[n], and for some frames it lands arbitrarily close to zero; the
    // dB (a logarithm) then amplifies the fp32 FFT's round-off without bound - 0.2 dB on one such frame moved VAD
    // probabilities by 4e-4 on long inputs (more frames, more near-zero draws; profiles/r2_precision.md). When the bin is
    // small against its neighbours (~2 % of the frame pairs) the group's 64 threads recompute it in double: n = j + 64 r
    // has the parity of j, so a thread's eight terms share one sign.
    if (j == 0) {
      const float2 zk = buf[grp][fft_idx(kNfft / 2)], z1 = buf[grp][fft_idx(kNfft / 2 - 1)], z2 = buf[grp][fft_idx(kNfft / 2 + 1)];
      const float scale = 0.02f * (fabsf(z1.x) + fabsf(z1.y) + fabsf(z2.x) + fabsf(z2.y));
      nyq_flag[grp] = ((va && fabsf(zk.x) < scale) ? 1 : 0) | ((vb && fabsf(zk.y) < scale) ? 2 : 0);
    }
    group_barrier(grp);
    if (nyq_flag[grp] != 0) {   // uniform over the group
      double sa = 0.0, sc = 0.0;
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        const int n = j + 64 * r;
        int64_t ia = (int64_t)ta * kHop + n - kNfft / 2, ib = ia + kHop;
        if (ia < 0) ia = -ia;
        if (ia >= L) ia = 2 * (L - 1) - ia;
        if (ib < 0) ib = -ib;
        if (ib >= L) ib = 2 * (L - 1) - ib;
        if (va) sa += (double)__ldg(xb + ia) * (double)win[n];
        if (vb) sc += (double)__ldg(xb + ib) * (double)win[n];
      }
      if (j & 1) { sa = -sa; sc = -sc; }
      sa = warp_sum(sa);
      sc = warp_sum(sc);
      if ((tid & 31) == 0) { nyq[grp][(tid >> 5) & 1][0] = sa; nyq[grp][(tid >> 5) & 1][1] = sc; }
      group_barrier(grp);
    }
    const bool wa = va && la >= 1 && la <= kFrontFrames;  // frames this CTA owns (not halo)
    const bool wb = vb && (la + 1) <= kFrontFrames;
    float2* Sa = S + ((int64_t)b * T + ta) * kBins;        // row of frame a; frame b is the next row
    float2* Sb = Sa + kBins;
    for (int f = j; f < kBins; f += 64) {
      float2 A = make_float2(0.f, 0.f), Bc = A;
      if (f > 0) {
        const float2 zk = buf[grp][fft_idx(f)], zn = buf[grp][fft_idx((kNfft - f) & (kNfft - 1))];
        A = make_float2(0.5f * (zk.x + zn.x), 0.5f * (zk.y - zn.y));
        Bc = make_float2(0.5f * (zk.y + zn.y), 0.5f * (zn.x - zk.x));
        if (f == kNfft / 2) {
          if (nyq_flag[grp] & 1) A.x = (float)(nyq[grp][0][0] + nyq[grp][1][0]);
          if (nyq_flag[grp] & 2) Bc.x = (float)(nyq[grp][0][1] + nyq[grp][1][1]);
        }
      }
      // lg2.approx (2^-22 relative on a value of at most ~100 dB) instead of the ~30-instruction log10f
      if (va) P[la][f + 1] = 10.f * __log10f(fmaxf(A.x * A.x + A.y * A.y, 1e-10f));
      if (vb) P[la + 1][f + 1] = 10.f * __log10f(fmaxf(Bc.x * Bc.x + Bc.y * Bc.y, 1e-10f));
      if (wa) Sa[f] = A;
      if (wb) Sb[f] = Bc;
    }
    __syncthreads();  // buf is rewritten by the next round
  }

  // activity gate; kernel index [i][j]: i over frequency, j over time (the input plane is [257, T]). A thread owns bin
  // tid + 1 (thread 0 also the DC bin) and walks the CTA's frames with a sliding 3 x 3 window: three shared-memory loads
  // per frame instead of nine.
  float s = 0.f, ss = 0.f;
  {
    const int nfr = min(kFrontFrames, T - t0);
    const int fcol = tid + 1;                      // column of P: [0] = bin -1 (zero), [f + 1] = bin f
    float k[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) k[i] = gk.k[i];
    // window w[jj][i] = P[lf - 1 + jj][fcol + i], jj = time tap, i = frequency tap
    float w0[3], w1[3], w2[3], d0[3], d1[3], d2[3];   // bins tid .. tid + 2 around bin tid + 1; d*: bins -1 .. 1 around the DC bin
#pragma unroll
    for (int i = 0; i < 3; ++i) { w0[i] = P[0][fcol + i]; w1[i] = P[1][fcol + i]; d0[i] = P[0][i]; d1[i] = P[1][i]; }
    float* zrow = z0 + ((int64_t)b * T + t0) * kC + tid;
    float* srow = SPECTRUM ? spectrum + ((int64_t)b * kBins + tid + 1) * T + t0 : nullptr;
    for (int lf = 1; lf <= nfr; ++lf) {
#pragma unroll
      for (int i = 0; i < 3; ++i) w2[i] = P[lf + 1][fcol + i];
      float z = w1[1];
      if (gk.enabled) {
        float acc = gk.bias;
#pragma unroll
        for (int i = 0; i < 3; ++i) acc += k[i * 3] * w0[i] + k[i * 3 + 1] * w1[i] + k[i * 3 + 2] * w2[i];
        z *= prelu(acc, gk.slope);
      }
      zrow[(int64_t)(lf - 1) * kC] = z;
      if constexpr (SPECTRUM) srow[lf - 1] = z;   // the optional torch-layout export (model.py:421)
      s += z;
      ss += z * z;
      if (tid == 0) {
#pragma unroll
        for (int i = 0; i < 3; ++i) d2[i] = P[lf + 1][i];
        float zd = d1[1];
        if (gk.enabled) {
          float acc = gk.bias;
#pragma unroll
          for (int i = 0; i < 3; ++i) acc += k[i * 3] * d0[i] + k[i * 3 + 1] * d1[i] + k[i * 3 + 2] * d2[i];
          zd *= prelu(acc, gk.slope);
        }
        const int64_t row = (int64_t)b * T + t0 + lf - 1;
        dc_gated[row] = zd;
        if constexpr (SPECTRUM) spectrum[((int64_t)b * kBins) * T + t0 + lf - 1] = zd;
#pragma unroll
        for (int i = 0; i < 3; ++i) { d0[i] = d1[i]; d1[i] = d2[i]; }
      }
#pragma unroll
      for (int i = 0; i < 3; ++i) { w0[i] = w1[i]; w1[i] = w2[i]; }
    }
  }
  block_stat_atomic(s, ss, st0 + b, red);
}

void launch_frontend(const float* x, int B, int64_t L, int T, const float* window, const float2* twiddle, int enabled,
                     const float* k3x3, float bias, float slope, float2* S, float* z0, float* dc_gated, Stat2* st0,
                     float* spectrum, cudaStream_t st) {
  GateK gk;
  for (int i = 0; i < 9; ++i) gk.k[i] = k3x3[i];  // Conv2d weight [1,1,3,3]: k[i*3+j], i = frequency tap, j = time tap
  gk.bias = bias;
  gk.slope = slope;
  gk.enabled = enabled;
  dim3 grid((T + kFrontFrames - 1) / kFrontFrames, B);
  // first kernel of the chain: it follows a memset, so it is launched without the PDL attribute
  if (spectrum != nullptr) launch_k(k_frontend<true>, grid, dim3(256), 0, st, false, x, L, T, window, twiddle, gk, S, z0, dc_gated, st0, spectrum);
  else launch_k(k_frontend<false>, grid, dim3(256), 0, st, false, x, L, T, window, twiddle, gk, S, z0, dc_gated, st0, spectrum);
}

}  // namespace septfa
