// Live streaming sessions (septfa_live_*): the kernels around the forward of one push.
// Every entry e of a push names a slot; the slot's hop counter k (hops its current stream has pushed so far) decides
// what the entry reads. Per slot the session keeps the last two input hops and the last two emitted hops (both
// speakers) in rings: hop k lives at ring position k & 1, so nothing is ever shifted.
// Reference: the 2 s left zero padding of model/online_class_known_targets.py:92-93 and the unknown-targets stitch of
// model/online_class_unknown_targets.py:84-94 (PITLossWrapper('pw_pt') with nn.L1Loss, n_src = 2, reorder, append).
#include "kernels.h"

namespace septfa {

constexpr int kLiveHop = 16000;
constexpr int kLiveWin = 3 * kLiveHop;
constexpr int kLiveVadFrame0 = 125;   // first window frame centred on the new hop: 125 * 256 = 2 hops
constexpr int kLiveVadFrames = 63;

// win[e] = concat(hop k-2, hop k-1, hop k) of entry e's stream, zeros for hops before the stream's first; then the new
// hop k takes ring position k & 1, where hop k-2 was. Each thread reads that element before it overwrites it.
__global__ void __launch_bounds__(256) k_live_window(const int32_t* __restrict__ slots, const int32_t* __restrict__ hops_done,
                                                     float* __restrict__ in_ring, const float* __restrict__ hops,
                                                     float* __restrict__ win) {
  const int e = blockIdx.y;
  const int slot = slots[e];
  const int k = hops_done[slot];
  float* ring = in_ring + (size_t)slot * 2 * kLiveHop;
  float* oldest = ring + (k & 1) * kLiveHop;              // hop k-2, replaced by hop k
  const float* prev = ring + ((k + 1) & 1) * kLiveHop;    // hop k-1
  const float* x = hops + (size_t)e * kLiveHop;
  float* w = win + (size_t)e * kLiveWin;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < kLiveHop; i += gridDim.x * blockDim.x) {
    const float v = x[i];
    w[i] = k >= 2 ? oldest[i] : 0.f;
    w[kLiveHop + i] = k >= 1 ? prev[i] : 0.f;
    w[2 * kLiveHop + i] = v;
    oldest[i] = v;
  }
}

void launch_live_window(const int32_t* slots, int n, const int32_t* hops_done, float* in_ring, const float* hops, float* win,
                        cudaStream_t st) {
  k_live_window<<<dim3(16, n), 256, 0, st>>>(slots, hops_done, in_ring, hops, win);
  ++ctx().launches;
}

// One CTA per entry. L1 PIT of the window prediction against what the stream already emitted, then the emit:
//   k = 0   pred[1 s, 2 s) against pred[2 s, 3 s) (the reference compares the first window with its own last second)
//   k = 1   pred[1 s, 2 s) against emitted hop 0
//   k >= 2  pred[0 s, 2 s) against emitted hops k-2, k-1
// |a - b| in fp32, sums in fp64; identity unless the swap is strictly cheaper (torch.min: the first index wins ties).
// The emitted hop k goes to tail ring position k & 1, over hop k-2, which the PIT has finished reading by then.
__global__ void __launch_bounds__(256) k_live_pit_emit(const int32_t* __restrict__ slots, int32_t* __restrict__ hops_done,
                                                       const float* __restrict__ pred, const float* __restrict__ vad, int T,
                                                       float* __restrict__ tail_ring, float* __restrict__ out,
                                                       float* __restrict__ out_vad, int32_t* __restrict__ perm) {
  __shared__ double red[4][8];
  __shared__ int s_swap;
  const int e = blockIdx.x;
  const int slot = slots[e];
  const int k = hops_done[slot];
  const float* p0 = pred + (size_t)e * 2 * kLiveWin;
  const float* p1 = p0 + kLiveWin;
  float* tail = tail_ring + (size_t)slot * 4 * kLiveHop;   // [2 positions][2 speakers][hop]
  const int nb = k >= 2 ? 2 : 1;                           // overlap in hops
  double v00 = 0.0, v01 = 0.0, v10 = 0.0, v11 = 0.0;
  for (int j = 0; j < nb; ++j) {
    const int pb = 2 - nb + j;   // window block compared with emitted hop k - nb + j
    const float4* a0 = reinterpret_cast<const float4*>(p0 + pb * kLiveHop);
    const float4* a1 = reinterpret_cast<const float4*>(p1 + pb * kLiveHop);
    const float* t = k == 0 ? nullptr : tail + ((k - nb + j) & 1) * 2 * kLiveHop;
    const float4* b0 = reinterpret_cast<const float4*>(k == 0 ? p0 + 2 * kLiveHop : t);
    const float4* b1 = reinterpret_cast<const float4*>(k == 0 ? p1 + 2 * kLiveHop : t + kLiveHop);
    for (int i = threadIdx.x; i < kLiveHop / 4; i += blockDim.x) {
      const float4 x0 = a0[i], x1 = a1[i], y0 = b0[i], y1 = b1[i];
      v00 += (double)fabsf(x0.x - y0.x) + (double)fabsf(x0.y - y0.y) + (double)fabsf(x0.z - y0.z) + (double)fabsf(x0.w - y0.w);
      v01 += (double)fabsf(x0.x - y1.x) + (double)fabsf(x0.y - y1.y) + (double)fabsf(x0.z - y1.z) + (double)fabsf(x0.w - y1.w);
      v10 += (double)fabsf(x1.x - y0.x) + (double)fabsf(x1.y - y0.y) + (double)fabsf(x1.z - y0.z) + (double)fabsf(x1.w - y0.w);
      v11 += (double)fabsf(x1.x - y1.x) + (double)fabsf(x1.y - y1.y) + (double)fabsf(x1.z - y1.z) + (double)fabsf(x1.w - y1.w);
    }
  }
  v00 = warp_sum(v00); v01 = warp_sum(v01); v10 = warp_sum(v10); v11 = warp_sum(v11);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) { red[0][w] = v00; red[1][w] = v01; red[2][w] = v10; red[3][w] = v11; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double s[4] = {0.0, 0.0, 0.0, 0.0};
    for (int q = 0; q < 4; ++q)
      for (int i = 0; i < 8; ++i) s[q] += red[q][i];
    const int sw = (s[0] + s[3]) <= (s[2] + s[1]) ? 0 : 1;
    s_swap = sw;
    perm[e * 2 + 0] = sw;
    perm[e * 2 + 1] = 1 - sw;
    hops_done[slot] = k + 1;   // read by the next push only: no other CTA of this push touches the slot
  }
  __syncthreads();
  const int sw = s_swap;
  const float* src0 = (sw ? p1 : p0) + 2 * kLiveHop;
  const float* src1 = (sw ? p0 : p1) + 2 * kLiveHop;
  float* t = tail + (k & 1) * 2 * kLiveHop;
  float* o = out + (size_t)e * 2 * kLiveHop;
  for (int i = threadIdx.x; i < kLiveHop; i += blockDim.x) {
    const float a = src0[i], b = src1[i];
    o[i] = a;
    o[kLiveHop + i] = b;
    t[i] = a;
    t[kLiveHop + i] = b;
  }
  if (out_vad)
    for (int i = threadIdx.x; i < 2 * kLiveVadFrames; i += blockDim.x) {
      const int spk = i / kLiveVadFrames, f = i - spk * kLiveVadFrames;
      out_vad[(size_t)e * 2 * kLiveVadFrames + i] = vad[((size_t)e * 2 + (spk ^ sw)) * T + kLiveVadFrame0 + f];
    }
}

void launch_live_pit_emit(const int32_t* slots, int n, int32_t* hops_done, const float* pred, const float* vad, int T,
                          float* tail_ring, float* out, float* out_vad, int32_t* perm, cudaStream_t st) {
  k_live_pit_emit<<<n, 256, 0, st>>>(slots, hops_done, pred, vad, T, tail_ring, out, out_vad, perm);
  ++ctx().launches;
}

// The slot list travels as a kernel argument (no device buffer, so releases on any stream cannot race on one).
struct LiveSlotChunk {
  int32_t n;
  int32_t id[kLiveReleaseChunk];
};

__global__ void k_live_release(LiveSlotChunk c, int32_t* __restrict__ hops_done) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < c.n) hops_done[c.id[i]] = 0;
}

void launch_live_release(const int32_t* slots_host, int n, int32_t* hops_done, cudaStream_t st) {
  for (int i0 = 0; i0 < n; i0 += kLiveReleaseChunk) {
    LiveSlotChunk c;
    c.n = n - i0 < kLiveReleaseChunk ? n - i0 : kLiveReleaseChunk;
    for (int i = 0; i < c.n; ++i) c.id[i] = slots_host[i0 + i];
    k_live_release<<<(c.n + 255) / 256, 256, 0, st>>>(c, hops_done);
    ++ctx().launches;
  }
}

}  // namespace septfa
