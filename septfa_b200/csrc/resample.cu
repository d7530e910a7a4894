// Resampling on the device: torchaudio.functional.resample(x, rate, 16000) with its defaults (sinc_interp_hann,
// lowpass_filter_width = 6, rolloff = 0.99), as read_mixture applies it through transforms.Resample, and the output
// direction resample(y, 16000, rate) with the same defaults. The two differ only in which side is the source: below,
// "native" samples are the source's (the rate's for kToModel, 16 kHz for kFromModel).
//
// With g = gcd(rate, 16000), orig = source / g and new = destination / g, output sample m = b new + p (phase p) is
//   y[m] = sum_j x[b orig + j - width] k[p][j],   j = 0 .. 2 width + orig - 1,   x = 0 outside [0, L),
// width = ceil(6 orig / base), base = 0.99 min(orig, new), and k[p][j] the Hann-windowed sinc at the scaled time
// t = base ((j - width) / orig - p / new). The bank keeps only the taps with |t| < 6 (beyond that torchaudio clamps t to
// +-6 and its taps are ~1e-20 or smaller); for each phase they are one contiguous run of j. The condition is decided in
// exact integer arithmetic (99 min(orig, new) |(j - width) new - p orig| < 600 orig new), so the support does not depend
// on rounding. The taps are computed in double in torchaudio's operation order and stored as fp32.
//
// resample_one() computes one output sample: an fp32 FMA chain over the phase's taps in increasing order, starting
// from 0. The batch kernel and the live kernel both call it on the same input values, so they give the same bits.
#include <algorithm>
#include <cmath>
#include <numeric>

#include "kernels.h"

namespace septfa {

namespace {

int64_t floor_div(int64_t a, int64_t b) {   // b > 0
  const int64_t q = a / b;
  return (a % b != 0 && a < 0) ? q - 1 : q;
}
int64_t ceil_div(int64_t a, int64_t b) { return -floor_div(-a, b); }

}  // namespace

bool resample_plan(int rate, ResampleDir dir, ResamplePlan* pl, std::vector<float>* taps, std::vector<int2>* spans) {
  if (rate < kResampleMinRate || rate > kResampleMaxRate) return false;
  ResamplePlan P{};
  if (rate == kResampleRate) {
    // torchaudio returns the input unchanged; one unit tap per output does the same (the int16 path converts with it)
    P.orig = P.nw = 1;
    P.ntaps = 1;
    P.tile_span = kResampleTile;
    if (taps) taps->assign(1, 1.f);
    if (spans) spans->assign(1, make_int2(0, 1));
    *pl = P;
    return true;
  }
  const int g = std::gcd(rate, kResampleRate);
  const int src = dir == kToModel ? rate : kResampleRate, dst = dir == kToModel ? kResampleRate : rate;
  const int64_t orig = src / g, nw = dst / g, mn = std::min(orig, nw);
  const double base = (double)mn * 0.99;
  const int64_t width = (int64_t)std::ceil(6.0 * (double)orig / base);
  // |t| < 6  <=>  (p orig 99 mn - 600 orig new) < c (99 mn new) < (p orig 99 mn + 600 orig new), c = j - width
  const int64_t A = 99 * mn * nw, K = 600 * orig * nw;
  std::vector<int64_t> cmin(nw), cmax(nw);
  int ntaps = 0;
  for (int64_t p = 0; p < nw; ++p) {
    const int64_t Bp = 99 * mn * p * orig;
    cmin[p] = std::max(floor_div(Bp - K, A) + 1, -width);
    cmax[p] = std::min(ceil_div(Bp + K, A) - 1, width + orig - 1);
    ntaps = std::max(ntaps, (int)(cmax[p] - cmin[p] + 1));
  }
  // D: output m = b new + p reads native samples up to b orig + cmax[p]. At N hops (N H a multiple of new), an output
  // q new - p samples before N H with cmax[p] >= q orig still needs a sample at or after N Hn.
  int64_t D = 0;
  for (int64_t p = 0; p < nw; ++p)
    if (cmax[p] >= orig) D = std::max(D, floor_div(cmax[p], orig) * nw - p);
  // history: the outputs of a push start at m = N H - D; the earliest native sample they read lies hist samples before
  // N Hn (the first sample of each phase increases with m, so outputs N H - D .. N H + new - 1 bound it)
  int64_t hist = 0;
  for (int64_t m = -D; m < nw; ++m) {
    const int64_t b = floor_div(m, nw), p = m - b * nw;
    hist = std::max(hist, -(b * orig + cmin[p]));
  }
  // staged native samples of a tile of kResampleTile consecutive outputs (periodic in its first output, period new)
  int64_t span = 0;
  for (int64_t p0 = 0; p0 < nw; ++p0) {
    const int64_t m1 = p0 + kResampleTile - 1, b1 = floor_div(m1, nw);
    span = std::max(span, b1 * orig + cmax[m1 - b1 * nw] - cmin[p0] + 1);
  }
  P.orig = (int)orig;
  P.nw = (int)nw;
  P.ntaps = ntaps;
  P.delay = (int)D;
  P.hist = (int)hist;
  P.tile_span = (int)span;
  if (spans) {
    spans->resize(nw);
    for (int64_t p = 0; p < nw; ++p) (*spans)[p] = make_int2((int)cmin[p], (int)(cmax[p] - cmin[p] + 1));
  }
  if (taps) {
    // torchaudio's _get_sinc_resample_kernel in float64: t = (-p / new + c / orig) * base, clamped to +-6; Hann window
    // cos(t pi / 6 / 2)^2; sinc(pi t) (1 at t = 0); times window * base / orig
    const double scale = base / (double)orig;
    taps->assign((size_t)nw * ntaps, 0.f);
    for (int64_t p = 0; p < nw; ++p)
      for (int64_t c = cmin[p]; c <= cmax[p]; ++c) {
        double t = ((double)(-p) / (double)nw + (double)c / (double)orig) * base;
        t = std::min(std::max(t, -6.0), 6.0);
        const double wcos = std::cos(t * M_PI / 6.0 / 2.0);
        const double win = wcos * wcos;
        t *= M_PI;
        double k = t == 0.0 ? 1.0 : std::sin(t) / t;
        k *= win * scale;
        (*taps)[(size_t)(c - cmin[p]) * nw + p] = (float)k;
      }
  }
  *pl = P;
  return true;
}

namespace {

__device__ __forceinline__ int64_t dev_floor_div(int64_t a, int64_t b) {
  const int64_t q = a / b;
  return (a % b != 0 && a < 0) ? q - 1 : q;
}

// A tile of outputs m0 .. m0 + n - 1 is addressed from its first output m0 = b0 new + p0: output m0 + t has phase
// p = (p0 + t) mod new and reads its taps from native sample lo + off, lo the first sample m0 reads. Only m0 needs
// 64-bit arithmetic; the rest stays in 32 bits.
__device__ __forceinline__ int64_t tile_first_input(const ResampleBank& bk, int64_t m0, int* p0) {
  const int64_t b0 = dev_floor_div(m0, bk.nw);
  *p0 = (int)(m0 - b0 * bk.nw);
  return b0 * bk.orig + bk.span[*p0].x;
}
__device__ __forceinline__ int tile_offset(const ResampleBank& bk, int p0, int t, int* p) {
  const int q = p0 + t, db = q / bk.nw;
  *p = q - db * bk.nw;
  return db * bk.orig + bk.span[*p].x - bk.span[p0].x;
}
// native samples a tile of n outputs reads, from lo on
__device__ __forceinline__ int tile_inputs(const ResampleBank& bk, int p0, int n) {
  int p;
  const int off = tile_offset(bk, p0, n - 1, &p);
  return off + bk.span[p].y;
}

// One output sample of phase p; x points at the first native sample it reads (taps are [ntaps][new], so the lanes of a
// warp, on consecutive phases, read consecutive taps).
__device__ __forceinline__ float resample_one(const ResampleBank& bk, int p, const float* x) {
  const int n = bk.span[p].y;
  const float* w = bk.taps + p;
  float acc = 0.f;
#pragma unroll 4
  for (int i = 0; i < n; ++i) acc = fmaf(x[i], __ldg(w + (size_t)i * bk.nw), acc);
  return acc;
}

// One CTA per tile of kResampleTile outputs of one row: the native samples the tile reads are staged in shared memory
// (converted to fp32; zeros outside [0, L)), then each thread computes outputs from there.
template <typename XT>
__global__ void __launch_bounds__(256) k_resample(const XT* __restrict__ x, int64_t L, int64_t L16, float* __restrict__ out,
                                                  ResampleBank bk) {
  extern __shared__ float xs[];
  const int64_t m0 = (int64_t)blockIdx.x * kResampleTile;
  const int nout = (int)min((int64_t)kResampleTile, L16 - m0);
  int p0;
  const int64_t lo = tile_first_input(bk, m0, &p0);
  const int n = tile_inputs(bk, p0, nout);
  const XT* xr = x + (size_t)blockIdx.y * L;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const int64_t gi = lo + i;
    xs[i] = (gi >= 0 && gi < L) ? (float)xr[gi] : 0.f;
  }
  __syncthreads();
  float* o = out + (size_t)blockIdx.y * L16 + m0;
  for (int t = threadIdx.x; t < nout; t += blockDim.x) {
    int p;
    const int off = tile_offset(bk, p0, t, &p);
    o[t] = resample_one(bk, p, xs + off);
  }
}

// Live sessions at a native rate: entry e (grid row) pushes hop k of the stream in slot slots[e]: Hn native samples,
// stream samples [k Hn, (k + 1) Hn). It writes u[k H, (k + 1) H) of u = concat(D zeros, resample(stream)) into
// u_out[e] and keeps the hop's last `hist` native samples for the next push. The history is double-buffered by the
// parity of k (push k reads buffer k & 1 and writes (k + 1) & 1), so CTAs of one row never race, and a push that fails
// after this kernel leaves the buffer the repeated push reads intact. A stream at k = 0 reads no history: its samples
// before 0 are zeros.
__global__ void __launch_bounds__(256) k_live_resample(const int32_t* __restrict__ slots, const int32_t* __restrict__ hops_done,
                                                       float* __restrict__ hist, const float* __restrict__ hops,
                                                       float* __restrict__ u_out, ResampleBank bk, int H, int Hn) {
  extern __shared__ float xs[];
  const int e = blockIdx.y;
  const int slot = slots[e];
  const int k = hops_done[slot];
  const int Hr = bk.hist;
  const int t0 = blockIdx.x * kResampleTile;
  const int nout = min(kResampleTile, H - t0);
  const int64_t m0 = (int64_t)k * H + t0 - bk.delay;       // y index of the tile's first output (< 0: before D)
  const int64_t kn = (int64_t)k * Hn;                        // stream index of the hop's first sample
  const float* x = hops + (size_t)e * Hn;
  const float* hr = hist + ((size_t)slot * 2 + (k & 1)) * Hr;
  int p0;
  const int64_t lo = tile_first_input(bk, m0, &p0);
  const int n = tile_inputs(bk, p0, nout);
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const int64_t gi = lo + i;
    xs[i] = gi < 0 ? 0.f : gi >= kn ? x[gi - kn] : hr[gi - (kn - Hr)];
  }
  __syncthreads();
  float* u = u_out + (size_t)e * H + t0;
  for (int t = threadIdx.x; t < nout; t += blockDim.x) {
    int p;
    const int off = tile_offset(bk, p0, t, &p);
    u[t] = m0 + t < 0 ? 0.f : resample_one(bk, p, xs + off);
  }
  if (blockIdx.x == 0) {
    float* hw = hist + ((size_t)slot * 2 + ((k + 1) & 1)) * Hr;
    for (int i = threadIdx.x; i < Hr; i += blockDim.x) hw[i] = x[Hn - Hr + i];
  }
}

// Live sessions at an output rate: grid row 2 e + c resamples channel c of entry e's emitted 16 kHz hop y[e][c] (stream
// samples [k H, (k + 1) H) of the channel, in the emitted speaker order) into out[e][c] = z[k Ho, (k + 1) Ho) of
// z = concat(D zeros, resample(y, 16000, rate)). It runs after k_live_pit_emit, which has advanced the slot's counter,
// so this push is k = hops_done - 1. The history [slot][parity][channel][hist] holds the channel's last `hist` 16 kHz
// samples, double-buffered by the parity of k as in k_live_resample; a stream at k = 0 reads none of it.
__global__ void __launch_bounds__(256) k_live_out_resample(const int32_t* __restrict__ slots,
                                                           const int32_t* __restrict__ hops_done, float* __restrict__ hist,
                                                           const float* __restrict__ y, float* __restrict__ out,
                                                           ResampleBank bk, int H, int Ho) {
  extern __shared__ float xs[];
  const int e = blockIdx.y >> 1, c = blockIdx.y & 1;
  const int slot = slots[e];
  const int k = hops_done[slot] - 1;
  const int Hr = bk.hist;
  const int t0 = blockIdx.x * kResampleTile;
  const int nout = min(kResampleTile, Ho - t0);
  const int64_t m0 = (int64_t)k * Ho + t0 - bk.delay;      // z index of the tile's first output (< 0: before D)
  const int64_t kh = (int64_t)k * H;                         // stream index of the hop's first sample
  const float* x = y + (size_t)blockIdx.y * H;
  const float* hr = hist + (((size_t)slot * 2 + (k & 1)) * 2 + c) * Hr;
  int p0;
  const int64_t lo = tile_first_input(bk, m0, &p0);
  const int n = tile_inputs(bk, p0, nout);
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const int64_t gi = lo + i;
    xs[i] = gi < 0 ? 0.f : gi >= kh ? x[gi - kh] : hr[gi - (kh - Hr)];
  }
  __syncthreads();
  float* o = out + (size_t)blockIdx.y * Ho + t0;
  for (int t = threadIdx.x; t < nout; t += blockDim.x) {
    int p;
    const int off = tile_offset(bk, p0, t, &p);
    o[t] = m0 + t < 0 ? 0.f : resample_one(bk, p, xs + off);
  }
  if (blockIdx.x == 0) {
    float* hw = hist + (((size_t)slot * 2 + ((k + 1) & 1)) * 2 + c) * Hr;
    for (int i = threadIdx.x; i < Hr; i += blockDim.x) hw[i] = x[H - Hr + i];
  }
}

}  // namespace

int64_t resample_out_len(const ResamplePlan& pl, int64_t L) { return ceil_div(L * pl.nw, pl.orig); }

void launch_resample(const void* x, bool pcm16, int B, int64_t L, int64_t L16, float* out, const ResampleBank& bk,
                     cudaStream_t st) {
  const dim3 grid((unsigned)((L16 + kResampleTile - 1) / kResampleTile), B);
  const size_t smem = (size_t)bk.tile_span * sizeof(float);
  if (pcm16)
    k_resample<int16_t><<<grid, 256, smem, st>>>(static_cast<const int16_t*>(x), L, L16, out, bk);
  else
    k_resample<float><<<grid, 256, smem, st>>>(static_cast<const float*>(x), L, L16, out, bk);
  ++ctx().launches;
}

void launch_live_resample(const int32_t* slots, int n, const int32_t* hops_done, float* hist, const float* hops, float* u,
                          const ResampleBank& bk, int H, int Hn, cudaStream_t st) {
  const dim3 grid((H + kResampleTile - 1) / kResampleTile, n);
  k_live_resample<<<grid, 256, (size_t)bk.tile_span * sizeof(float), st>>>(slots, hops_done, hist, hops, u, bk, H, Hn);
  ++ctx().launches;
}

void launch_live_out_resample(const int32_t* slots, int n, const int32_t* hops_done, float* hist, const float* y, float* out,
                              const ResampleBank& bk, int H, int Ho, cudaStream_t st) {
  const dim3 grid((Ho + kResampleTile - 1) / kResampleTile, 2 * n);
  k_live_out_resample<<<grid, 256, (size_t)bk.tile_span * sizeof(float), st>>>(slots, hops_done, hist, y, out, bk, H, Ho);
  ++ctx().launches;
}

}  // namespace septfa
