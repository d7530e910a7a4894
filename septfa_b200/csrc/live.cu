// Live streaming sessions (septfa_live_*): the kernels around the forward of one push.
// Every entry e of a push names a slot; the slot's hop counter k (hops its current stream has pushed so far) decides
// what the entry reads. A session has a window of W samples and a hop of H samples (R = W - H). Per slot it keeps the
// last R input samples and the last R emitted samples (both speakers) in rings: stream sample s lives at ring position
// s mod R, so nothing is ever shifted.
// Reference: the left zero padding of model/online_class_known_targets.py:92-93 and the unknown-targets stitch of
// model/online_class_unknown_targets.py:84-94 (PITLossWrapper('pw_pt') with nn.L1Loss, n_src = 2, reorder, append).
#include "kernels.h"

namespace septfa {

// win[e] = concat(the stream's samples [kH - R, kH), zeros before its first sample; the new hop). Window position
// i < R holds stream sample kH - R + i, at ring position (kH + i) mod R; for i < H that is where element i of the new
// hop goes, so the thread that reads a ring element is the one that overwrites it (2 H <= W: positions i >= H are only
// read).
__global__ void __launch_bounds__(256) k_live_window(const int32_t* __restrict__ slots, const int32_t* __restrict__ hops_done,
                                                     float* __restrict__ in_ring, const float* __restrict__ hops,
                                                     float* __restrict__ win, LiveGeom g) {
  const int e = blockIdx.y;
  const int slot = slots[e];
  const int k = hops_done[slot];
  const int H = g.hop, R = g.win - g.hop;
  const int64_t kh = (int64_t)k * H;
  const int base = (int)(kh % R);                        // ring position of stream sample kH
  const int first = kh >= R ? 0 : R - (int)kh;           // window positions below this precede the stream
  float* ring = in_ring + (size_t)slot * R;
  const float* x = hops + (size_t)e * H;
  float* w = win + (size_t)e * g.win;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < R; i += gridDim.x * blockDim.x) {
    int p = base + i;
    if (p >= R) p -= R;
    w[i] = i >= first ? ring[p] : 0.f;
    if (i < H) {
      const float v = x[i];
      w[R + i] = v;
      ring[p] = v;
    }
  }
}

void launch_live_window(const int32_t* slots, int n, const int32_t* hops_done, float* in_ring, const float* hops, float* win,
                        LiveGeom g, cudaStream_t st) {
  k_live_window<<<dim3(16, n), 256, 0, st>>>(slots, hops_done, in_ring, hops, win, g);
  ++ctx().launches;
}

// One CTA per entry. L1 PIT of the window prediction against what the stream already emitted, then the emit:
//   k = 0   pred[R - H, R) against pred[R, W) (the reference compares the first window with its own last hop)
//   k >= 1  pred[R - o, R) against the last o = min(kH, R) emitted samples
// The overlap is summed one emitted hop at a time, oldest first (the oldest is partial when H does not divide R), each
// hop in float4 steps strided over the CTA: |a - b| in fp32, sums in fp64, so the order is fixed (and at W = 3 H it is
// that of the earlier two-hop-ring kernel). Identity unless the swap is strictly cheaper (torch.min: the first index
// wins ties). The emitted hop overwrites the ring positions of samples [kH - R, kH - R + H), which the PIT has finished
// reading at the block barrier.
__global__ void __launch_bounds__(256) k_live_pit_emit(const int32_t* __restrict__ slots, int32_t* __restrict__ hops_done,
                                                       const float* __restrict__ pred, const float* __restrict__ vad, int T,
                                                       float* __restrict__ tail_ring, float* __restrict__ out,
                                                       float* __restrict__ out_vad, int32_t* __restrict__ perm, LiveGeom g) {
  __shared__ double red[4][8];
  __shared__ int s_swap;
  const int e = blockIdx.x;
  const int slot = slots[e];
  const int k = hops_done[slot];
  const int W = g.win, H = g.hop, R = g.win - g.hop;
  const int64_t kh = (int64_t)k * H;
  const int base = (int)(kh % R);                          // ring position of stream sample kH
  const float* p0 = pred + (size_t)e * 2 * W;
  const float* p1 = p0 + W;
  float* tail = tail_ring + (size_t)slot * 2 * R;          // [2 speakers][R]
  const int ov = k == 0 ? H : (int)min(kh, (int64_t)R);   // overlap in samples
  double v00 = 0.0, v01 = 0.0, v10 = 0.0, v11 = 0.0;
  for (int dhi = ov; dhi > 0;) {                           // samples dhi .. dlo + 1 before kH: one emitted hop
    const int dlo = (dhi - 1) / H * H;
    const int n4 = (dhi - dlo) >> 2;
    const float4* a0 = reinterpret_cast<const float4*>(p0 + R - dhi);
    const float4* a1 = reinterpret_cast<const float4*>(p1 + R - dhi);
    int t0 = base - dhi;                                   // ring position of stream sample kH - dhi
    if (t0 < 0) t0 += R;
    for (int i = threadIdx.x; i < n4; i += blockDim.x) {
      const float4 x0 = a0[i], x1 = a1[i];
      float4 y0, y1;
      if (k == 0) {
        y0 = reinterpret_cast<const float4*>(p0 + W - dhi)[i];
        y1 = reinterpret_cast<const float4*>(p1 + W - dhi)[i];
      } else {
        int q = t0 + 4 * i;
        if (q >= R) q -= R;
        y0 = *reinterpret_cast<const float4*>(tail + q);
        y1 = *reinterpret_cast<const float4*>(tail + R + q);
      }
      v00 += (double)fabsf(x0.x - y0.x) + (double)fabsf(x0.y - y0.y) + (double)fabsf(x0.z - y0.z) + (double)fabsf(x0.w - y0.w);
      v01 += (double)fabsf(x0.x - y1.x) + (double)fabsf(x0.y - y1.y) + (double)fabsf(x0.z - y1.z) + (double)fabsf(x0.w - y1.w);
      v10 += (double)fabsf(x1.x - y0.x) + (double)fabsf(x1.y - y0.y) + (double)fabsf(x1.z - y0.z) + (double)fabsf(x1.w - y0.w);
      v11 += (double)fabsf(x1.x - y1.x) + (double)fabsf(x1.y - y1.y) + (double)fabsf(x1.z - y1.z) + (double)fabsf(x1.w - y1.w);
    }
    dhi = dlo;
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
  const float* src0 = (sw ? p1 : p0) + R;
  const float* src1 = (sw ? p0 : p1) + R;
  float* o = out + (size_t)e * 2 * H;
  for (int i = threadIdx.x; i < H; i += blockDim.x) {
    int q = base + i;
    if (q >= R) q -= R;
    const float a = src0[i], b = src1[i];
    o[i] = a;
    o[H + i] = b;
    tail[q] = a;
    tail[R + q] = b;
  }
  if (out_vad) {
    const int F = g.vad_frames;
    for (int i = threadIdx.x; i < 2 * F; i += blockDim.x) {
      const int spk = i / F, f = i - spk * F;
      out_vad[(size_t)e * 2 * F + i] = vad[((size_t)e * 2 + (spk ^ sw)) * T + g.vad_frame0 + f];
    }
  }
}

void launch_live_pit_emit(const int32_t* slots, int n, int32_t* hops_done, const float* pred, const float* vad, int T,
                          float* tail_ring, float* out, float* out_vad, int32_t* perm, LiveGeom g, cudaStream_t st) {
  k_live_pit_emit<<<n, 256, 0, st>>>(slots, hops_done, pred, vad, T, tail_ring, out, out_vad, perm, g);
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
