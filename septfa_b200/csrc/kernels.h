// Host-side launcher declarations shared by the septfa translation units.
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <vector>
#include "common.cuh"

namespace septfa {

// ---- parameters of the three dense contractions (shared by the tcgen05 and the fp32 engines)

// Residual-stream affine: y = (w - mean_b) * rstd_b * gamma[c] + beta[c]; gamma == nullptr means y = w.
struct StreamNorm {
  const Stat2* st;     // [B] accumulators of the producing stage (ignored if gamma == nullptr)
  const float* gamma;  // [256]
  const float* beta;   // [256]
  float eps;
  double inv_n;        // 1 / (256 * T)
};

// DepthConv1d first half (model/model.py:132/138): p = PReLU(W1 y + b1), stats of p.
struct Conv1Params {
  const float* w_in;   // [M,256] residual stream (pre-norm)
  StreamNorm norm;
  int M, T, B;
  const float* bias;   // [256]
  float slope;
  const __half* w_img; // tcgen05 image of W1*diag(gamma_in): 4 K-chunks x [256 rows x 128 B], 128B-swizzled K-major
  const float* bias_f; // [256] b1 + W1 beta_in (the stream norm's affine folded into the weights; tcgen05 engine)
  const float* w_t;    // fp32 [256 k][256 n]
  void* p_out;         // [M,256] fp32, or fp16 when half_io
  Stat2* st_p;         // [B]
  int half_io;         // store p as fp16 (both conv1 and dconv on the tcgen05 engine)
  int planes = 0;      // store p (fp16) as K-group planes [32][Mp][8] for the tensor-core depthwise kernel (dconv_mma2.cu)
  int Mp = 0;          // slots per plane; frame r lives in slot r + kPlaneHalo
  const __half* w_img_lo = nullptr;  // low part of the fp16 weight split ("accurate" precision mode)
  int split = 0;       // split-precision operands: three tensor-core passes, fp32-accurate contraction
};

// DepthConv1d second half (model/model.py:136/142,144) with GroupNorm reg2 folded into W3:
// q = PReLU(dconv(GN1(p))), racc = (W3*diag(g2)) q  (raw accumulators), row/column sums of racc.
struct DconvParams {
  const void* p_in;    // [M,256] fp32, or fp16 when half_io
  const Stat2* st_p;   // [B]
  const float* g1;     // reg1 gamma/beta [256]
  const float* be1;
  const float4* w2b;   // [512] {w[o][0], w[o][1], w[o][2], b2[o]}
  const float4* w2f;   // [512] reg1 folded in: {w[o][k]*g1[o/2] (k=0..2), their sum}
  const float* c2f;    // [512] b2[o] + be1[o/2] * sum_k w[o][k]
  float slope2;
  int dil;
  int M, T, B;
  const __half* w_img; // 8 K-chunks x [256 rows x 128 B]
  const float* w_t;    // fp32 [512 k][256 n] (gamma2-folded)
  void* racc;          // [M,256] fp32, or fp16 when half_io
  float* rowsum;       // [M]
  double* colsum;      // [B,256] (pre-zeroed, accumulated with double atomics)
  Stat2* st_q;         // [B]
  int half_io;         // p and racc are fp16
  const float4* wtab;  // tcgen05 engine: the folded taps in pair order, 640 float4 (septfa_abi.cu: dconv tap table)
  const float* bog;    // tcgen05 engine: [256] beta1 / gamma1 (zero-padding substitute, see gemm_tc.cu)
  const __half* w_img_lo = nullptr;  // low part of the fp16 weight split ("accurate" precision mode)
  int split = 0;       // split-precision operands: three tensor-core passes, fp32-accurate contraction
};

// Plane layout of p for dconv_mma2.cu: [32 K-groups of 8 channels][Mp slots][8 halves], frame r in slot r + kPlaneHalo;
// the kPlaneHalo slots in front of frame 0 and the slots behind frame M - 1 are zero.
constexpr int kPlaneHalo = 4;                      // = the largest dilation
constexpr int kDconvTapBytes = 16 * 3 * 1024;      // [16 channel groups][3 taps][32 outputs x 16 inputs, fp16]
struct DconvMmaParams {
  const __half* p_planes; int Mp;
  const Stat2* st_p;
  const uint8_t* tap_img2;  // block-diagonal tap matrices split along the outputs into the two halves a CTA pair holds
  const float4* swc;        // [256] {sw[2i], sw[2i+1], c2f[2i], c2f[2i+1]}: sums of the fp16 taps, folded constants
  const float* w16;         // [3][512] the fp16-rounded folded taps as fp32
  const float* bog;         // [256] beta1 / gamma1
  float slope2; int dil;
  int M, T, B;
  const __half* w_img;      // res_out image, as DconvParams
  __half* racc; float* rowsum; double* colsum; Stat2* st_q;
  const void* racc_tmap = nullptr;   // host pointer to a CUtensorMap over racc ([M rows][256 halves], box 64 x 32, SWIZZLE_128B)
  int discard = 0;          // drop the consumed lines of p from the L2 (discard.global.L2)
};

// TCN.output (model/model.py:322-325,357): logits = Wo GN(PReLU(y)) + bo, N = 514 padded to 576.
struct OutConvParams {
  const float* w_in;   // [M,256]
  StreamNorm norm;
  float slope_o;
  const Stat2* st_o;   // [B] stats of PReLU(y)
  const float* g_o;    // output.1 gamma/beta [256], eps 1e-5
  const float* b_o;
  int M, T, B;
  const float* bias;   // [576] (zero padded)
  const __half* w_img; // 3 N-tiles x 4 K-chunks x [192 rows x 128 B]: high part of the fp16 split
  const __half* w_img_lo; // low part: fp16(w - fp16(w))
  const float* w_t;    // fp32 [256 k][576 n]
  float* logits;       // [M,576]
};

// TF_Attention scalars (model/model.py:182-208).
struct TfParams {
  float wt1[3], bt1, wt2[3], bt2, at;
  float wf1[3], bf1, wf2[3], bf2, af;
  int enabled;
};

// r[c,t] = racc[t,c] * ra[b] + rb[b,c];  residual = r * gf[b,c] * gt[row]
struct GateParams {
  const Stat2* st_q;   // [B], over 512*T elements, eps 1e-8
  const float* s3;     // [256] sum_o W3g[c,o]
  const float* c03;    // [256] sum_o W3[c,o]*beta2[o] + b3[c]
  const float* rowsum; // [M]
  const double* colsum; // [B,256]
  TfParams tf;
  int M, T, B;
  float* ra;           // [B]
  float* rb;           // [B,256]
  float* gf;           // [B,256]
  float* gt;           // [M]
  float* mt;           // [M] scratch of the streaming gate kernel: per-frame channel means
};

enum LnMode { LN_NONE = 0, LN_RECURSIVE = 1, LN_RESIDUAL = 2 };

struct ResidParams {
  float* w;            // [M,256] residual stream, updated in place by resid_apply
  StreamNorm norm;     // affine that turns w into y
  const void* racc;    // [M,256] fp32, or fp16 when racc_half
  int racc_half;
  const float* ra; const float* rb; const float* gf; const float* gt;
  int M, T, B;
  int mode;            // LnMode
  Stat2* st_v;         // [B] stats of v (y + r*g for recursive, r*g for residual)
  const float* g_a;    // ln_first (recursive) or ln_modules (residual) gamma/beta, eps 1e-5
  const float* b_a;
  Stat2* st_w;         // [B] stats of the new stream (recursive only)
  const __half* w_half_in = nullptr;   // half-stream mode (cluster-resident kernel only): the stream before the block as fp16 ...
  __half* w_half_out = nullptr;        // ... and after it; a null pointer means the fp32 buffer `w`
  int discard = 0;                     // cluster-resident kernel: drop the consumed lines of racc from the L2
};

// ---- launchers ---------------------------------------------------------------------------
// frontend.cu
void make_twiddles(float2* host256);
void launch_frontend(const float* x, int B, int64_t L, int T, const float* window, const float2* twiddle, int enabled,
                     const float* k3x3, float bias, float slope, float2* S, float* z0, float* dc_gated, Stat2* st0,
                     float* spectrum /*optional [B,257,T] export, nullable*/, cudaStream_t st);
// tcn.cu
void launch_ref_conv1(const Conv1Params& p, cudaStream_t st);
void launch_ref_dconv(const DconvParams& p, cudaStream_t st);
void launch_ref_outconv(const OutConvParams& p, cudaStream_t st);
void launch_tf_gate(const GateParams& p, cudaStream_t st);
void launch_resid_stats(const ResidParams& p, cudaStream_t st);
void launch_resid_apply(const ResidParams& p, cudaStream_t st);
void launch_out_stats(const float* w, StreamNorm norm, float slope, int M, int T, Stat2* st_o, cudaStream_t st);
// resid_fused.cu: gates + both residual GroupNorm steps in one cluster-resident kernel
cudaError_t resid_fused_setup();
int resid_fused_cluster_size(int T);   // 0: the utterance does not fit one cluster
// clusters of the kernel variant (stream read / written as fp16) the device keeps resident at once (occupancy query)
int resid_fused_resident_clusters(bool in_half, bool out_half, int T);
// launches min(clusters, B) clusters of resid_fused_cluster_size(T) CTAs; racc is fp16
void launch_resid_fused(const ResidParams& rp, const GateParams& gp, int clusters, cudaStream_t st);
// preproc.cu
void launch_minmax_normalize(const float* x, int B, int64_t L, const int64_t* lengths /*nullable*/, unsigned* ext /*[B][2] scratch*/,
                             float* out, cudaStream_t st);
void launch_minmax_normalize_pcm16(const int16_t* x, int B, int64_t L, const int64_t* lengths /*nullable*/, unsigned* ext, float* out,
                                   cudaStream_t st);
void launch_to_half(const float* in, __half* out, int64_t n, cudaStream_t st);
void launch_sisdr(const float* p, const float* t, int64_t rows, int64_t n, int zero_mean, double* scratch /*[rows][5]*/, float* out,
                  cudaStream_t st);
// gemm_conv1_tma.cu: conv1 of the half-stream mode (the stream is the fp16 A operand itself, fed by TMA tensor loads)
struct Conv1TmaParams {
  const void* a_tmap;       // host pointer to a CUtensorMap over the fp16 stream [M rows][256], box 64 x 128, SWIZZLE_128B
  StreamNorm norm;          // statistics of the stream (gamma == nullptr: y = w); the affine is folded into w_img / sb
  int M, T, B;
  const __half* w_img;      // W1 * diag(gamma_in) image
  const float4* sb;         // [128] {S[2i], S[2i+1], b'[2i], b'[2i+1]}: row sums of the fp16 image, folded bias
  float slope;
  __half* p_planes; int Mp;
  Stat2* st_p;
};
cudaError_t conv1_tma_setup();
void launch_conv1_tma(const Conv1TmaParams& p, cudaStream_t st);
// gemm_conv1_pair.cu: conv1 on CTA pairs with TF32 operands (the fp32 stream is the A operand itself, fed by TMA; weights resident)
struct Conv1PairParams {
  const void* a_tmap;       // host pointer to a CUtensorMap over the fp32 stream [M rows][256], box 32 x 128, SWIZZLE_128B
  StreamNorm norm;          // statistics of the stream (gamma == nullptr: y = w); the affine is folded into w_img / sb
  int M, T, B;
  const float* w_img;       // TF32 image of W1 * diag(gamma_in): 8 K-chunks x [256 rows x 128 B]
  const float4* sb;         // [128] {S[2i], S[2i+1], b'[2i], b'[2i+1]}: row sums of the TF32 image, folded bias
  float slope;
  __half* p_planes; int Mp;
  Stat2* st_p;
};
cudaError_t conv1_pair_setup();
void launch_conv1_pair(const Conv1PairParams& p, cudaStream_t st);
// gemm_conv1_persist.cu
cudaError_t conv1_persist_setup();
void launch_conv1_persist(const Conv1Params& p, cudaStream_t st);   // fp16 p (half_io), T >= 128
// dconv_mma2.cu: tensor-core depthwise + res_out kernel on CTA pairs (cta_group::2) with the weights resident in shared memory
cudaError_t dconv_mma2_setup();
void launch_dconv_mma2(const DconvMmaParams& p, cudaStream_t st);
// gemm_tc.cu
void launch_tc_conv1(const Conv1Params& p, cudaStream_t st);
void launch_tc_dconv(const DconvParams& p, cudaStream_t st);
void launch_tc_outconv(const OutConvParams& p, cudaStream_t st);
cudaError_t tc_gemm_setup();  // opt-in shared memory attributes; call once per device
// backend.cu
struct VadParams {
  const float* logits;   // [M,576]; columns kVadCol0 + s*20 + k*4 + j hold the conv1_1 partial products (out conv)
  int M, T, B;
  float b1[4]; float slope; float g[4]; float be[4];
  float w2[12]; float b2;  // output_layer_vad [4 j][3 k]
  float* c4;             // [B*2*T, 4] scratch
  float* prob;           // [B,2,T]
  float* smooth;         // [B,2,T]
  float thr;
  int do_smooth;
};
void launch_vad(const VadParams& p, cudaStream_t st);
cudaError_t backend_setup();   // opt-in shared memory of the mask / iSTFT / export kernel; call once per device
void launch_mask_istft(const float2* S, const float* logits, const float* gate /*[B,2,T] or null*/, const float* window,
                       const float2* twiddle, int B, int64_t L, int T, float* out, cudaStream_t st);
// waveform [B,2,L]; the exports est [B,2,257,T] complex, mask [B,2,257,T], logits_out [B,514,T] are each nullable
void launch_mask_istft_export(const float2* S, const float* logits, const float* gate /*[B,2,T] or null*/, const float* window,
                              const float2* twiddle, int B, int64_t L, int T, float* out, float2* est, float* mask,
                              float* logits_out, cudaStream_t st);
// online.cu
void launch_pit(const float* a, int64_t a_bstride, int64_t a_sstride, const float* b, int64_t b_bstride, int64_t b_sstride,
                int S, int64_t n, double* acc /*[S,4] zeroed*/, int32_t* perm, cudaStream_t st);
void launch_online_emit(const float* pred /*[S,2,Lw]*/, int64_t Lw, const int32_t* perm, int S, int hop, int tail_cap,
                        const float* tail_in /*[S,2,tail_cap]*/, int tail_len, float* tail_out, float* emitted /*[S,2,hop]*/,
                        cudaStream_t st);
// live.cu: streaming sessions with a window of W and a hop of H samples (R = W - H). Slots index the per-slot state:
// hops_done [capacity], in_ring [capacity][R], tail_ring [capacity][2][R]; slots (device) [n] lists the slot of each
// entry of a push. The caller has checked the geometry: 256 <= H, 2 H <= W, W and H multiples of 16.
struct LiveGeom {
  int win, hop;               // W, H
  int vad_frame0, vad_frames; // j0 = ceil((W - H) / 256), F = ceil(W / 256) - j0
};
constexpr int kLiveReleaseChunk = 1000;   // slots per release launch (passed by value: 4 KB of kernel arguments)
void launch_live_window(const int32_t* slots, int n, const int32_t* hops_done, float* in_ring, const float* hops /*[n,H]*/,
                        float* win /*[n,W]*/, LiveGeom g, cudaStream_t st);
void launch_live_pit_emit(const int32_t* slots, int n, int32_t* hops_done, const float* pred /*[n,2,W]*/,
                          const float* vad /*[n,2,T]*/, int T, float* tail_ring, float* out /*[n,2,H]*/,
                          float* out_vad /*[n,2,F] or null*/, int32_t* perm /*[n,2]*/, LiveGeom g, cudaStream_t st);
void launch_live_release(const int32_t* slots_host, int n, int32_t* hops_done, cudaStream_t st);

// ---- resampling between 16 kHz and another rate (resample.cu)
constexpr int kResampleRate = 16000;
constexpr int kResampleMinRate = 8000, kResampleMaxRate = 192000;
constexpr int kResampleTile = 512;   // outputs per CTA
// Direction of a bank: a rate's input to the model's 16 kHz, or the model's 16 kHz output to a rate.
enum ResampleDir { kToModel = 0, kFromModel = 1 };
// What a rate needs, computed on the host from the bank's effective support. "Source" is the side the bank reads
// (the native rate for kToModel, 16 kHz for kFromModel), "destination" the side it writes.
struct ResamplePlan {
  int orig, nw;        // source / g, destination / g with g = gcd(rate, 16000)
  int ntaps;           // taps stored per phase (the longest effective run; shorter ones are zero-padded)
  int delay;           // D: destination samples a live stream lags by
  int hist;            // source samples a live push reads from before its hop
  int tile_span;       // source samples one tile of kResampleTile outputs reads (shared memory floats)
};
struct ResampleBank {
  const float* taps;   // [ntaps][nw] fp32, tap i of phase p at i * nw + p
  const int2* span;    // [nw] {first j - width, tap count} of each phase
  int orig, nw, delay, hist, tile_span;
};
// false for a rate outside [8000, 192000]; taps / spans (nullable) receive the bank
bool resample_plan(int rate, ResampleDir dir, ResamplePlan* plan, std::vector<float>* taps, std::vector<int2>* spans);
int64_t resample_out_len(const ResamplePlan& plan, int64_t L);   // ceil(nw L / orig)
void launch_resample(const void* x, bool pcm16, int B, int64_t L, int64_t L16, float* out, const ResampleBank& bk,
                     cudaStream_t st);
void launch_live_resample(const int32_t* slots, int n, const int32_t* hops_done, float* hist /*[cap][2][hist]*/,
                          const float* hops /*[n,Hn]*/, float* u /*[n,H]*/, const ResampleBank& bk, int H, int Hn,
                          cudaStream_t st);
// after launch_live_pit_emit (hops_done already advanced): y [n,2,H] at 16 kHz -> out [n,2,Ho] at the output rate
void launch_live_out_resample(const int32_t* slots, int n, const int32_t* hops_done, float* hist /*[cap][2][2][hist]*/,
                              const float* y, float* out, const ResampleBank& bk, int H, int Ho, cudaStream_t st);

// Per-handle launch state (septfa_handle owns one; every C-ABI entry binds it to the calling thread before launching).
// Which kernel runs at each stage of a forward is decided by plan_forward (septfa_abi.cu); the launchers only launch.
struct LaunchCtx {
  int launches = 0;            // kernels launched since the last reset (host counter)
  int use_pdl = 1;             // launch with the programmatic-stream-serialization attribute
  int sm_count = 0;            // SMs of the handle's device: the grids of the persistent and CTA-pair kernels
};
LaunchCtx& ctx();
void bind_ctx(LaunchCtx* c);

// Grid of a launch; cluster > 0 launches clusters of that many CTAs along x (for kernels without __cluster_dims__).
struct Grid {
  dim3 dim;
  unsigned cluster;
  Grid(dim3 d, unsigned cs = 0) : dim(d), cluster(cs) {}
};

// Kernel launch with (optional) programmatic dependent launch; counts the launch.
template <typename... KArgs, typename... Args>
inline void launch_k(void (*kern)(KArgs...), Grid grid, dim3 block, size_t smem, cudaStream_t st, bool pdl, Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid.dim;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[2];
  int n = 0;
  if (grid.cluster > 0) {
    at[n].id = cudaLaunchAttributeClusterDimension;
    at[n].val.clusterDim.x = grid.cluster; at[n].val.clusterDim.y = 1; at[n].val.clusterDim.z = 1;
    ++n;
  }
  if (pdl && ctx().use_pdl) {
    at[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
  }
  cfg.attrs = at;
  cfg.numAttrs = n;
  cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
  ++ctx().launches;
}

}  // namespace septfa
