// C ABI of libseptfa.so (include/septfa.h): handle, weight folding / packing, workspace carving,
// the forward pass orchestration and the online (sliding-window) step.
// Reference: model/model.py:360-461 (SeparationModel), model/online_class_unknown_targets.py:72-105.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include <cuda.h>

#include "../../include/septfa.h"
#include "kernels.h"

using namespace septfa;

namespace {

thread_local std::string g_create_error;

struct KeySpec {
  std::string name;
  int64_t numel;
};

struct DevBlock {
  const float* w1_img32; const float4* sb1_32;   // gemm_conv1_pair.cu: TF32 image of W1 diag(gamma), {row sums, folded bias}
  const float4* sb1;   // gemm_conv1_tma.cu: {S[2i], S[2i+1], b1f[2i], b1f[2i+1]}
  const __half* w1_img; const __half* w1_img_lo; const __half* w3_img_lo; const float* w1_t; const float* b1; const float* b1f; float a1; const float* g1; const float* be1;
  const float4* w2b; const float4* w2f; const float* c2f; float a2; int dil;
  const float4* wtab; const float* bog;   // tcgen05 dconv producer: pair-ordered tap table, beta1 / gamma1
  const uint8_t* tap_img2; const float4* swc; const float* w16; bool mma_ok;   // tensor-core depthwise kernel (dconv_mma2.cu)
  const __half* w3_img; const float* w3_t; const float* s3_tc; const float* s3_ref; const float* c03;
  TfParams tf;
  const float* lf_g; const float* lf_b; const float* ls_g; const float* ls_b;  // recursive
  const float* lm_g; const float* lm_b;                                        // residual
};

}  // namespace

struct septfa_handle {
  septfa_config cfg{};
  int device = 0;
  int nblk = 0;
  int ln_mode = LN_NONE;
  int engine = SEPTFA_ENGINE_TCGEN05_F16;
  bool committed = false;
  std::string err;
  std::vector<KeySpec> keys;
  std::map<std::string, std::vector<float>> host;
  std::vector<void*> allocs;
  // device weights
  std::vector<DevBlock> blocks;
  const float* ln_g = nullptr; const float* ln_b = nullptr;
  float out_a = 0.f; const float* out_g = nullptr; const float* out_be = nullptr;
  const __half* out_img = nullptr; const __half* out_img_lo = nullptr; const float* out_wt = nullptr; const float* out_bias = nullptr;
  float vad_b1[4]{}; float vad_a = 0.f; float vad_g[4]{}; float vad_be[4]{};
  float vad_w2[12]{}; float vad_b2 = 0.f;
  float act_k[9]{}; float act_b = 0.f; float act_a = 0.f;
  const float* win_fwd = nullptr; const float* win_inv = nullptr; const float2* twiddle = nullptr;
  int last_launches = 0;
  LaunchCtx lctx;   // launch options, device facts and counter of this handle (bound to the calling thread by every entry point)
  // forward_host resources
  cudaStream_t hstream = nullptr, hstream_in = nullptr, hstream_out = nullptr;
  cudaEvent_t hev_in[8] = {}, hev_done[8] = {};
  unsigned* norm_ext = nullptr; int norm_cap = 0;   // septfa_minmax_normalize scratch
  int host_chunks = 0;  // 0 = automatic
  struct HostSlot {      // septfa_forward_host_submit / _wait
    cudaStream_t stream = nullptr;          // copies of this slot
    cudaEvent_t ev_in = nullptr, ev_done = nullptr;
    float* x = nullptr; float* out = nullptr; float* vad = nullptr; void* ws = nullptr;
    void* xraw = nullptr; void* out16 = nullptr; unsigned* ext = nullptr;   // PCM16 input staging, fp16 output staging, extrema
    size_t cap_x = 0, cap_out = 0, cap_vad = 0, cap_ws = 0, cap_xraw = 0, cap_out16 = 0, cap_ext = 0;
    bool busy = false;
  } slots[SEPTFA_HOST_SLOTS];
  cudaStream_t slot_compute = nullptr;      // kernels of both slots, in submission order
  // kernel options (septfa_set_option), read by plan_forward
  int fused_resid = 1;    // cluster-resident gate + residual kernel when the utterance fits a cluster
  int precision = SEPTFA_PRECISION_AUTO;
  int conv1_persist = 1;  // persistent warp-specialised conv1 kernel (0: always the one-tile-per-CTA kernel)
  int conv1_pair = 1;     // blocks 1 .. n-1, recursive-LN wiring, fast mode: TF32 CTA-pair conv1 fed by TMA from the fp32 stream
                          // (1: from ~2.5 tiles per SM on, 2: always)
  int stream_half = 0;    // opt-in: blocks 1 .. n-1 carry the residual stream as fp16 (recursive-LN wiring, fast precision
                          // mode). 11 % faster, but the stream's rounding random-walks through all blocks: worst VAD
                          // error on the shape sweep 9.5e-4 against 2.1e-4 - outside the default parity envelope
  int dconv_mma = 1;      // tensor-core depthwise + res_out kernel on CTA pairs (dconv_mma2.cu) when applicable
  int l2_discard = 1;     // consumed hand-off buffers (p in the pair dconv kernel, racc in the cluster residual kernel) are discarded from the L2
  // resident clusters of the cluster residual kernel by (variant, frame count): an occupancy query of this handle's
  // device, cached so that a forward does not repeat it (a cache: filling it changes no plan)
  mutable std::map<std::pair<int, int>, int> resid_clusters;
  bool all_mma_ok = false;                 // every block's folded taps are representable for the tensor-core depthwise kernel
  float* hx_dev = nullptr; float* hout_dev = nullptr; float* hvad_dev = nullptr; void* hws = nullptr; void* hws_b = nullptr;
  float* hx_pin = nullptr; float* hout_pin = nullptr; float* hvad_pin = nullptr;
  size_t hcap_x = 0, hcap_out = 0, hcap_vad = 0, hcap_ws = 0, hcap_ws_b = 0;
  // pit scratch
  double* pit_acc = nullptr; int pit_cap = 0;
  // optional per-kernel-class profiling (CUDA events recorded on the launch stream)
  int profile = 0;
  std::vector<cudaEvent_t> ev_pool;
  std::vector<int> ev_cat;   // category of the interval that STARTS at event i
  int ev_used = 0;
  double prof_ms[SEPTFA_PROF_NCAT] = {0};
  int prof_launches[SEPTFA_PROF_NCAT] = {0};
  // resampling filter banks by (direction, rate), and their device memory: kept apart from `allocs`, which a weight
  // commit frees, since live sessions and later calls hold the bank pointers until septfa_destroy
  std::map<std::pair<int, int>, ResampleBank> banks;
  std::vector<void*> bank_allocs;
};

struct septfa_graph {
  septfa_handle* h = nullptr;
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  int nodes = 0, kernels = 0;
};

struct septfa_online {
  septfa_handle* h = nullptr;
  int S = 0;
  int win = 0, hop = 0;   // W, H; the emitted tail keeps the last W - H samples
  int hops = 0;
  int tail_len = 0;
  int cur = 0;
  float* tail[2] = {nullptr, nullptr};
  double* acc = nullptr;
};

struct septfa_live {
  septfa_handle* h = nullptr;
  int capacity = 0;
  LiveGeom g{};                   // window W, hop H, VAD frames j0 .. j0 + F - 1
  int32_t* hops_done = nullptr;   // [capacity] hops pushed by the slot's current stream (0: no history is read)
  float* in_ring = nullptr;       // [capacity][W - H] the last W - H input samples, sample s at position s mod (W - H)
  float* tail_ring = nullptr;     // [capacity][2][W - H] the last W - H emitted samples of both speakers, the same way
  int rate = kResampleRate;       // input rate; other than 16000: each push is resampled first
  int in_hop = 0;                 // Hn = H rate / 16000 native samples per push
  ResampleBank bank{};            // the handle's bank for `rate`
  float* hist = nullptr;          // [capacity][2][bank.hist] native history, double-buffered by hop parity
  int out_rate = kResampleRate;   // output rate; other than 16000: each emitted hop is resampled last
  int out_hop = 0;                // Ho = H out_rate / 16000 output samples per push
  ResampleBank out_bank{};        // the handle's 16000 -> out_rate bank
  float* hist_out = nullptr;      // [capacity][2 parity][2 channels][out_bank.hist] 16 kHz history of the emitted channels
};

namespace {

constexpr int kFs = 16000, kWinLen = 48000, kHopLen = 16000;
constexpr int kMaxWinLen = 160000;   // 10 s
constexpr int kHostChunksMax = 8;

int fail(septfa_handle* h, int code, const std::string& msg) {
  if (h) h->err = msg; else g_create_error = msg;
  return code;
}

// Window W and hop H of an online state or a live session: 256 <= H, 2 H <= W <= 160000, both multiples of 16 (1 ms,
// so that ring segments and float4 accesses stay aligned).
int check_geometry(septfa_handle* h, int W, int H) {
  const std::string g = "window " + std::to_string(W) + ", hop " + std::to_string(H) + ": ";
  if (H < 256) return fail(h, SEPTFA_E_INVALID, g + "the hop must be >= 256 samples");
  if (W < 2 * (int64_t)H) return fail(h, SEPTFA_E_INVALID, g + "the window must be >= 2 hops");
  if (W > kMaxWinLen) return fail(h, SEPTFA_E_INVALID, g + "the window must be <= 160000 samples (10 s)");
  if (W % 16 || H % 16) return fail(h, SEPTFA_E_INVALID, g + "window and hop must be multiples of 16 samples (1 ms)");
  return 0;
}

// An input or output rate the resampler accepts: an integer in [8000, 192000] Hz.
int check_rate(septfa_handle* h, int rate, ResampleDir dir, ResamplePlan* plan) {
  if (!resample_plan(rate, dir, plan, nullptr, nullptr))
    return fail(h, SEPTFA_E_INVALID, dir == kToModel
                    ? "rate " + std::to_string(rate) + ": the input rate must lie in 8000 .. 192000 Hz"
                    : "out rate " + std::to_string(rate) + ": the output rate must lie in 8000 .. 192000 Hz");
  return 0;
}

#define CUDA_TRY(h, expr)                                                                     \
  do {                                                                                        \
    cudaError_t e_ = (expr);                                                                  \
    if (e_ != cudaSuccess)                                                                    \
      return fail(h, SEPTFA_E_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_));      \
  } while (0)

void add_wn_conv(std::vector<KeySpec>& k, const std::string& p, int co, int ci, int ks) {
  k.push_back({p + ".bias", co});
  k.push_back({p + ".weight_g", co});
  k.push_back({p + ".weight_v", (int64_t)co * ci * ks});
}
void add_gn(std::vector<KeySpec>& k, const std::string& p, int c) {
  k.push_back({p + ".weight", c});
  k.push_back({p + ".bias", c});
}

// Key families and shapes of the reference state_dict (SURVEY.md section 8b; model/model.py:210-325,153-171,376-400).
void build_keys(septfa_handle* h) {
  auto& k = h->keys;
  const auto& c = h->cfg;
  k.push_back({"spec_input.spec.window", 512});
  k.push_back({"spec_output.window", 512});
  k.push_back({"inv_spec.window", 512});
  add_gn(k, "TCN.LN", kC);
  for (int i = 0; i < h->nblk; ++i) {
    const std::string p = "TCN.TCN." + std::to_string(i);
    add_wn_conv(k, p + ".conv1d", kC, kC, 1);
    add_wn_conv(k, p + ".dconv1d", kH, 1, 3);
    add_wn_conv(k, p + ".res_out", kC, kH, 1);
    k.push_back({p + ".nonlinearity1.weight", 1});
    k.push_back({p + ".nonlinearity2.weight", 1});
    add_gn(k, p + ".reg1", kC);
    add_gn(k, p + ".reg2", kH);
  }
  if (c.tf_attention)
    for (int i = 0; i < h->nblk; ++i) {
      const std::string p = "TCN.time_freq_attnetion." + std::to_string(i);  // (sic) model.py:279
      for (const char* n : {"conv1d_t_1", "conv1d_t_2", "conv1d_f_1", "conv1d_f_2"}) {
        k.push_back({p + "." + n + ".weight", 3});
        k.push_back({p + "." + n + ".bias", 1});
      }
      k.push_back({p + ".prelu_t.weight", 1});
      k.push_back({p + ".prelu_f.weight", 1});
    }
  if (c.apply_recursive_ln)
    for (int i = 0; i < h->nblk; ++i) {
      add_gn(k, "TCN.ln_first_modules." + std::to_string(i), kC);
      add_gn(k, "TCN.ln_second_modules." + std::to_string(i), kC);
    }
  if (c.apply_residual_ln)
    for (int i = 0; i < h->nblk; ++i) add_gn(k, "TCN.ln_modules." + std::to_string(i), kC);
  k.push_back({"TCN.output.0.weight", 1});
  add_gn(k, "TCN.output.1", kC);
  add_wn_conv(k, "TCN.output.2", kBins * 2, kC, 1);
  if (c.final_vad) {
    add_wn_conv(k, "vad.common.conv1_1", 4, kBins, 5);
    k.push_back({"vad.common.relu_1.weight", 1});
    add_gn(k, "vad.common.BN_1", 4);
    add_wn_conv(k, "vad.output_layer_vad", 1, 4, 3);
  }
  if (c.activity_input_bool) {
    k.push_back({"activity_input.weight", 9});
    k.push_back({"activity_input.bias", 1});
    k.push_back({"prelu.weight", 1});
  }
}

// torch.nn.utils.weight_norm (dim 0): w[o,:] = g[o] * v[o,:] / ||v[o,:]||_2  (model.py:104-127,159-163,324)
std::vector<double> fold_wn(const std::vector<float>& g, const std::vector<float>& v, int co) {
  const size_t per = v.size() / co;
  std::vector<double> w(v.size());
  for (int o = 0; o < co; ++o) {
    double n2 = 0.0;
    for (size_t i = 0; i < per; ++i) n2 += (double)v[o * per + i] * (double)v[o * per + i];
    const double sc = (double)g[o] / std::sqrt(n2);
    for (size_t i = 0; i < per; ++i) w[o * per + i] = sc * (double)v[o * per + i];
  }
  return w;
}

template <typename T>
int upload(septfa_handle* h, const std::vector<T>& src, const T** dst) {
  void* d = nullptr;
  CUDA_TRY(h, cudaMalloc(&d, src.size() * sizeof(T)));
  h->allocs.push_back(d);
  CUDA_TRY(h, cudaMemcpy(d, src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice));
  *dst = reinterpret_cast<const T*>(d);
  return 0;
}

// The handle's bank for `rate` in direction `dir` (checked by the caller), built and uploaded at the first call for
// them. The upload is waited for, so the bank can be used on any stream afterwards; later calls find it in the cache.
int get_bank(septfa_handle* h, int rate, ResampleDir dir, cudaStream_t st, ResampleBank* out) {
  const std::pair<int, int> key{(int)dir, rate};
  auto it = h->banks.find(key);
  if (it != h->banks.end()) { *out = it->second; return 0; }
  ResamplePlan pl{};
  std::vector<float> taps;
  std::vector<int2> spans;
  resample_plan(rate, dir, &pl, &taps, &spans);
  float* dt = nullptr;
  int2* ds = nullptr;
  CUDA_TRY(h, cudaMalloc(reinterpret_cast<void**>(&dt), taps.size() * sizeof(float)));
  h->bank_allocs.push_back(dt);
  CUDA_TRY(h, cudaMalloc(reinterpret_cast<void**>(&ds), spans.size() * sizeof(int2)));
  h->bank_allocs.push_back(ds);
  CUDA_TRY(h, cudaMemcpyAsync(dt, taps.data(), taps.size() * sizeof(float), cudaMemcpyHostToDevice, st));
  CUDA_TRY(h, cudaMemcpyAsync(ds, spans.data(), spans.size() * sizeof(int2), cudaMemcpyHostToDevice, st));
  CUDA_TRY(h, cudaStreamSynchronize(st));
  const ResampleBank bk{dt, ds, pl.orig, pl.nw, pl.delay, pl.hist, pl.tile_span};
  h->banks[key] = bk;
  *out = bk;
  return 0;
}

// tcgen05 operand image of W[n][k] (n < nrows_valid, K = kdim): tiles of NT rows, K-chunks of 64 halves,
// each chunk = NT rows x 128 B, K-major with the 128-byte swizzle (16-byte chunk index XOR row%8).
std::vector<__half> pack_image(const std::vector<double>& w, int nvalid, int kdim, int ntiles, int NT) {
  const int nch = kdim / 64;
  std::vector<__half> img((size_t)ntiles * nch * NT * 64, __float2half(0.f));
  for (int tile = 0; tile < ntiles; ++tile)
    for (int j = 0; j < nch; ++j)
      for (int r = 0; r < NT; ++r) {
        const int n = tile * NT + r;
        if (n >= nvalid) continue;
        for (int kk = 0; kk < 64; ++kk) {
          const int k = j * 64 + kk;
          const size_t byte = ((size_t)(tile * nch + j) * NT) * 128 + (size_t)(r >> 3) * 1024 + (size_t)(r & 7) * 128 +
                              (size_t)(((kk >> 3) ^ (r & 7)) << 4) + (size_t)(kk & 7) * 2;
          img[byte / 2] = __float2half((float)w[(size_t)n * kdim + k]);
        }
      }
  return img;
}

// Low part of the 2-term fp16 split of a weight matrix: w - fp16(w), evaluated on the fp32 value.
std::vector<double> split_lo(const std::vector<double>& w) {
  std::vector<double> lo(w.size());
  for (size_t i = 0; i < w.size(); ++i) lo[i] = (double)((float)w[i] - __half2float(__float2half((float)w[i])));
  return lo;
}

// CUtensorMap over the fp16 residual stream [rows][256]: box = 64 halves x 128 rows with the 128-byte swizzle, i.e. one
// K-chunk of a 128-frame tile lands in shared memory as a K-major SWIZZLE_128B tcgen05 operand (rows past `rows`: zeros).
bool make_stream_tmap(CUtensorMap* out, const void* gptr, int64_t rows, int box_rows = 128, bool f32 = false) {
  typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                               const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                               CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static EncodeFn fn = nullptr;
  if (!fn) {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) != cudaSuccess || sym == nullptr) {
      cudaGetLastError();
      return false;
    }
    fn = reinterpret_cast<EncodeFn>(sym);
  }
  const cuuint64_t dims[2] = {(cuuint64_t)kC, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)kC * (f32 ? 4 : 2)};
  const cuuint32_t box[2] = {f32 ? 32u : 64u, (cuuint32_t)box_rows};   // 128-byte rows either way
  const cuuint32_t estr[2] = {1, 1};
  return fn(out, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(gptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

const std::vector<float>& T_(septfa_handle* h, const std::string& k) { return h->host.at(k); }

struct Workspace {
  float2* S; float* w; __half* wh; float* dcg; float* p; float* racc; float* rowsum; float* gt; float* mt; float* logits;
  float* ra; float* rb; float* gf; float* c4; float* prob; float* smooth;
  uint8_t* zero_begin; size_t zero_bytes;
  Stat2* st0; Stat2* st_blk; Stat2* st_o; Stat2* st_vad; double* colsum;
  size_t total;
};

Workspace carve(const septfa_handle* h, void* base, int B, int64_t L) {
  Workspace w{};
  const int64_t T = septfa_num_frames(L), M = (int64_t)B * T;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    uint8_t* p = reinterpret_cast<uint8_t*>(base) + off;
    off += (bytes + 255) & ~(size_t)255;
    return p;
  };
  w.S = (float2*)take(M * kBins * sizeof(float2));
  w.w = (float*)take(M * kC * sizeof(float));
  w.wh = (__half*)take(M * kC * sizeof(__half));   // the residual stream as fp16 (half-stream mode)
  w.dcg = (float*)take(M * sizeof(float));
  w.p = (float*)take(M * kC * sizeof(float) + (size_t)(256 + 2 * kPlaneHalo) * 512);   // also holds the fp16 plane layout (Mp slots)
  w.racc = (float*)take(M * kC * sizeof(float));
  w.rowsum = (float*)take(M * sizeof(float));
  w.gt = (float*)take(M * sizeof(float));
  w.mt = (float*)take(M * sizeof(float));
  w.logits = (float*)take(M * kLogitStride * sizeof(float));
  w.ra = (float*)take(B * sizeof(float));
  w.rb = (float*)take((size_t)B * kC * sizeof(float));
  w.gf = (float*)take((size_t)B * kC * sizeof(float));
  w.c4 = (float*)take(M * 2 * 4 * sizeof(float));
  w.prob = (float*)take(M * 2 * sizeof(float));
  w.smooth = (float*)take(M * 2 * sizeof(float));
  w.zero_begin = reinterpret_cast<uint8_t*>(base) + off;
  w.st0 = (Stat2*)take(B * sizeof(Stat2));
  w.st_blk = (Stat2*)take((size_t)h->nblk * 4 * B * sizeof(Stat2));
  w.st_o = (Stat2*)take(B * sizeof(Stat2));
  w.st_vad = (Stat2*)take((size_t)B * 2 * sizeof(Stat2));
  w.colsum = (double*)take((size_t)h->nblk * B * kC * sizeof(double));
  w.zero_bytes = (reinterpret_cast<uint8_t*>(base) + off) - w.zero_begin;
  w.total = off;
  return w;
}

// Record an event that starts an interval of category `cat` (cat < 0: closing event).
void prof_mark(septfa_handle* h, int cat, cudaStream_t st) {
  if (!h->profile) return;
  if (h->ev_used == (int)h->ev_pool.size()) {
    cudaEvent_t e;
    cudaEventCreate(&e);
    h->ev_pool.push_back(e);
    h->ev_cat.push_back(-1);
  }
  cudaEventRecord(h->ev_pool[h->ev_used], st);
  h->ev_cat[h->ev_used] = cat;
  ++h->ev_used;
}

int check_forward_args(septfa_handle* h, int B, int64_t L) {
  if (!h) return SEPTFA_E_INVALID;
  if (!h->committed) return fail(h, SEPTFA_E_STATE, "weights not committed");
  if (B < 1) return fail(h, SEPTFA_E_INVALID, "B must be >= 1");
  if (L < 257) return fail(h, SEPTFA_E_INVALID, "L must be >= 257 (reflect padding of 256 samples needs a longer input)");
  if (B > 32767) return fail(h, SEPTFA_E_INVALID, "B must be <= 32767 per call (grid limits): split larger batches, utterances are independent");
  if ((int64_t)B * septfa_num_frames(L) > (int64_t)1 << 30) return fail(h, SEPTFA_E_INVALID, "B*T too large");
  return 0;
}

// Which kernel runs at each stage of a forward, and the storage modes that tie neighbouring kernels together.
enum class Conv1Kernel { ref, tc_gemm, persist, pair, tma };
enum class DconvKernel { ref, tc_gemm, mma2 };
struct ForwardPlan {
  bool split;             // split-precision operands of conv1 / dconv ("accurate" mode): fp32 p / racc
  bool half_io;           // p and racc stored as fp16
  bool planes;            // p stored as K-group planes of Mp slots (written by the persistent / pair / TMA conv1, read by mma2)
  int Mp;
  bool stream_half;       // blocks 1 .. n-1 carry the residual stream as fp16
  Conv1Kernel conv1_first, conv1_rest;   // block 0, blocks 1 .. n-1
  DconvKernel dconv;
  int resid_clusters[2][2];   // [stream read as fp16][stream written as fp16]: resident clusters of the cluster residual
                              // kernel for the variants the forward runs; all 0: k_tf_gate + the streaming kernels
  bool tc_out;            // output conv on the tensor cores (else the fp32 CUDA-core kernel)
  bool exports;           // back end: k_mask_istft_export (any est / mask / logits export), else k_mask_istft
};

int resident_clusters(const septfa_handle& h, bool in_half, bool out_half, int T) {
  const auto key = std::make_pair((in_half ? 2 : 0) + (out_half ? 1 : 0), T);
  auto it = h.resid_clusters.find(key);
  if (it == h.resid_clusters.end()) it = h.resid_clusters.emplace(key, resid_fused_resident_clusters(in_half, out_half, T)).first;
  return it->second;
}

ForwardPlan plan_forward(const septfa_handle& h, int B, int64_t L, bool exports) {
  ForwardPlan pl{};
  const int T = (int)septfa_num_frames(L);
  const int64_t M = (int64_t)B * T;
  // engine is a bit mask of the contractions that run on the fp32 CUDA-core kernels
  const bool tc_conv1 = !(h.engine & 1), tc_dconv = !(h.engine & 2);
  pl.tc_out = !(h.engine & 4);
  // p (conv1 -> dconv) and racc (dconv -> residual kernels) are stored as fp16 when both producers run on the tensor
  // cores: their consumers round to fp16 operands anyway, and emulation on the oracle shows no change of the VAD /
  // waveform error (DESIGN.md section 3); the fp32 CUDA-core engine keeps fp32 storage.
  // Precision mode of the two block contractions: "accurate" = split-precision operands (three tensor-core passes) and
  // fp32 p / racc. AUTO picks it for the residual-LN wiring (config_without_vad): its stream is never re-normalised, so
  // the fp16 roundings of all 24 blocks accumulate to ~1e-3 in VAD probability, against ~1e-4 with the recursive-LN
  // wiring of config_with_vad (measured: DESIGN.md, "Precision").
  pl.split = tc_conv1 && tc_dconv &&
             (h.precision == SEPTFA_PRECISION_ACCURATE || (h.precision == SEPTFA_PRECISION_AUTO && h.ln_mode == LN_RESIDUAL));
  pl.half_io = tc_conv1 && tc_dconv && !pl.split;
  // Tensor-core depthwise kernel (dconv_mma2.cu): p travels as K-group planes, which only the persistent conv1 (and
  // the pair / TMA conv1 of blocks 1 .. n-1) write.
  const bool persist = pl.half_io && T >= 128 && h.conv1_persist;
  pl.planes = persist && h.dconv_mma && h.all_mma_ok;
  pl.Mp = (int)((M + 255) / 256 * 256 + 2 * kPlaneHalo);   // whole tile PAIRS (dconv_mma2.cu walks its tiles in pairs)
  // Gates + both residual GroupNorm steps in one cluster-resident kernel when an utterance fits a cluster and the
  // device keeps clusters of it resident.
  const bool fused = h.fused_resid && pl.half_io && resid_fused_cluster_size(T) > 0;
  // Half-stream mode: between the blocks the residual stream is stored as fp16 (written by the cluster-resident residual
  // kernel of block i, read by TMA as the A operand of conv1 of block i + 1 and by the residual kernel of block i + 1); the
  // first block reads the front end's fp32 features, the last block writes fp32 for the output layer. Recursive-LN wiring
  // in the fast precision mode only: the stream is re-normalised by every block, so its fp16 rounding is one more source of
  // the size of the operand roundings (DESIGN.md, "Precision"), and the residual-LN wiring runs the accurate mode anyway.
  // Only the cluster kernel reads and writes the fp16 stream, so every variant the blocks run must have resident clusters.
  if (fused && pl.planes && h.stream_half && h.ln_mode == LN_RECURSIVE && h.nblk > 1) {
    pl.resid_clusters[0][1] = resident_clusters(h, false, true, T);
    pl.resid_clusters[1][0] = resident_clusters(h, true, false, T);
    if (h.nblk > 2) pl.resid_clusters[1][1] = resident_clusters(h, true, true, T);
    pl.stream_half = pl.resid_clusters[0][1] > 0 && pl.resid_clusters[1][0] > 0 && (h.nblk == 2 || pl.resid_clusters[1][1] > 0);
    if (!pl.stream_half) pl.resid_clusters[0][1] = pl.resid_clusters[1][0] = pl.resid_clusters[1][1] = 0;
  }
  if (fused && !pl.stream_half) pl.resid_clusters[0][0] = resident_clusters(h, false, false, T);
  // TF32 CTA-pair conv1 (gemm_conv1_pair.cu) for blocks 1 .. n-1: the fp32 stream is its A operand, fetched by TMA
  // (from ~2.5 tiles per SM on: each of its CTAs first loads 128 KB of weights, which 1-2 tiles do not pay back - measured
  // at 64 / 128 / 256 x 4 s: +0.06 / +0.03 / -0.055 ms per forward against the persistent producer kernel; option value 2
  // forces it at any size)
  const bool pair = pl.planes && !pl.stream_half && h.conv1_pair && h.ln_mode == LN_RECURSIVE && h.nblk > 1 &&
                    (h.conv1_pair == 2 || (M + 127) / 128 * 2 >= (int64_t)h.lctx.sm_count * 5);
  pl.conv1_first = !tc_conv1 ? Conv1Kernel::ref : (persist ? Conv1Kernel::persist : Conv1Kernel::tc_gemm);
  pl.conv1_rest = pl.stream_half ? Conv1Kernel::tma : (pair ? Conv1Kernel::pair : pl.conv1_first);
  pl.dconv = pl.planes ? DconvKernel::mma2 : (tc_dconv ? DconvKernel::tc_gemm : DconvKernel::ref);
  // With any of the est / mask / logits exports, one kernel writes them and the waveform from one read of S and the logits;
  // without them the register-prefetch kernel (3 CTAs per SM against 2) is slightly faster end to end (DESIGN.md section 3).
  pl.exports = exports;
  return pl;
}

}  // namespace

extern "C" {

const char* septfa_version(void) { return "septfa-b200 0.1 (sm_100a)"; }

const char* septfa_last_error(const septfa_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int64_t septfa_num_frames(int64_t L) { return 1 + L / kHop; }

int septfa_create(septfa_handle** out, const septfa_config* cfg, int device) {
  if (!out || !cfg) return fail(nullptr, SEPTFA_E_INVALID, "null argument");
  *out = nullptr;
  const septfa_config& c = *cfg;
  // Configurations outside the shipped ones are rejected loudly (SURVEY.md section 8a, "unused-at-these-configs").
  if (c.n_fft_bins != 512 || c.bn_dim != 256 || c.h_dim != 512 || c.num_spk != 2)
    return fail(nullptr, SEPTFA_E_INVALID, "unsupported sizes: need n_fftBins=512, BN_dim=256, H_dim=512, num_spk=2");
  if (!c.weight_norm) return fail(nullptr, SEPTFA_E_INVALID, "unsupported config: weight_norm=false");
  if (c.skip) return fail(nullptr, SEPTFA_E_INVALID, "unsupported config: skip=true");
  if (!c.dilated) return fail(nullptr, SEPTFA_E_INVALID, "unsupported config: dilated=false");
  if (c.causal) return fail(nullptr, SEPTFA_E_INVALID, "unsupported config: casual=true (cLN)");
  if (c.final_vad_masked_speakers) return fail(nullptr, SEPTFA_E_INVALID, "unsupported config: final_vad_masked_speakers=true");
  if (c.layer < 1 || c.stack < 1 || c.layer * c.stack > 256) return fail(nullptr, SEPTFA_E_INVALID, "bad layer/stack");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(nullptr, SEPTFA_E_CUDA, "no CUDA device visible (this library has no CPU fallback)");
  if (device < 0 || device >= ndev) return fail(nullptr, SEPTFA_E_INVALID, "bad device index");
  cudaDeviceProp prop{};
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return fail(nullptr, SEPTFA_E_CUDA, "cudaGetDeviceProperties failed");
  if (prop.major != 10) return fail(nullptr, SEPTFA_E_CUDA, "device is not sm_100 (Blackwell B200); this build targets sm_100a only");
  auto* h = new septfa_handle();
  h->cfg = c;
  h->device = device;
  h->nblk = c.layer * c.stack;
  h->ln_mode = c.apply_recursive_ln ? LN_RECURSIVE : (c.apply_residual_ln ? LN_RESIDUAL : LN_NONE);  // model.py:347-352
  build_keys(h);
  if (cudaSetDevice(device) != cudaSuccess) { delete h; return fail(nullptr, SEPTFA_E_CUDA, "cudaSetDevice failed"); }
  cudaDeviceGetAttribute(&h->lctx.sm_count, cudaDevAttrMultiProcessorCount, device);
  cudaError_t e = tc_gemm_setup();
  if (e == cudaSuccess) e = resid_fused_setup();
  if (e == cudaSuccess) e = conv1_persist_setup();
  if (e == cudaSuccess) e = conv1_tma_setup();
  if (e == cudaSuccess) e = conv1_pair_setup();
  if (e == cudaSuccess) e = dconv_mma2_setup();
  if (e == cudaSuccess) e = backend_setup();
  if (e != cudaSuccess) { delete h; return fail(nullptr, SEPTFA_E_CUDA, std::string("tc_gemm_setup: ") + cudaGetErrorString(e)); }
  *out = h;
  return 0;
}

void septfa_destroy(septfa_handle* h) {
  if (!h) return;
  bind_ctx(nullptr);
  cudaSetDevice(h->device);
  for (void* p : h->allocs) cudaFree(p);
  for (void* p : h->bank_allocs) cudaFree(p);
  cudaFree(h->norm_ext);
  cudaFree(h->hx_dev); cudaFree(h->hout_dev); cudaFree(h->hvad_dev); cudaFree(h->hws); cudaFree(h->hws_b); cudaFree(h->pit_acc);
  if (h->slot_compute) { cudaStreamSynchronize(h->slot_compute); cudaStreamDestroy(h->slot_compute); }
  for (auto& sl : h->slots) {
    if (sl.stream) { cudaStreamSynchronize(sl.stream); cudaStreamDestroy(sl.stream); }
    if (sl.ev_in) cudaEventDestroy(sl.ev_in);
    if (sl.ev_done) cudaEventDestroy(sl.ev_done);
    cudaFree(sl.x); cudaFree(sl.out); cudaFree(sl.vad); cudaFree(sl.ws); cudaFree(sl.xraw); cudaFree(sl.out16); cudaFree(sl.ext);
  }
  cudaFreeHost(h->hx_pin); cudaFreeHost(h->hout_pin); cudaFreeHost(h->hvad_pin);
  if (h->hstream) {
    cudaStreamDestroy(h->hstream); cudaStreamDestroy(h->hstream_in); cudaStreamDestroy(h->hstream_out);
    for (int i = 0; i < kHostChunksMax; ++i) { cudaEventDestroy(h->hev_in[i]); cudaEventDestroy(h->hev_done[i]); }
  }
  for (cudaEvent_t e : h->ev_pool) cudaEventDestroy(e);
  delete h;
}

int septfa_num_keys(const septfa_handle* h) { return h ? (int)h->keys.size() : 0; }
const char* septfa_key_name(const septfa_handle* h, int i) {
  return (h && i >= 0 && i < (int)h->keys.size()) ? h->keys[i].name.c_str() : nullptr;
}
int64_t septfa_key_numel(const septfa_handle* h, int i) {
  return (h && i >= 0 && i < (int)h->keys.size()) ? h->keys[i].numel : -1;
}

int septfa_set_tensor(septfa_handle* h, const char* key, const float* data, int64_t numel) {
  if (!h || !key || !data) return SEPTFA_E_INVALID;
  for (const auto& k : h->keys)
    if (k.name == key) {
      if (k.numel != numel)
        return fail(h, SEPTFA_E_KEY, std::string("size mismatch for ") + key + ": expected " + std::to_string(k.numel) +
                                         " elements, got " + std::to_string(numel));
      h->host[key].assign(data, data + numel);
      h->committed = false;
      return 0;
    }
  return fail(h, SEPTFA_E_KEY, std::string("unexpected key ") + key);
}

int septfa_set_option(septfa_handle* h, const char* name, int value) {
  if (!h || !name) return SEPTFA_E_INVALID;
  if (std::strcmp(name, "engine") == 0) {
    if (value < 0 || value > 7) return fail(h, SEPTFA_E_INVALID, "bad engine");
    h->engine = value;
    return 0;
  }
  if (std::strcmp(name, "profile") == 0) {
    h->profile = value ? 1 : 0;
    return 0;
  }
  if (std::strcmp(name, "conv1_persist") == 0) {
    h->conv1_persist = value ? 1 : 0;
    return 0;
  }
  if (std::strcmp(name, "conv1_pair") == 0) {
    h->conv1_pair = value == 2 ? 2 : (value ? 1 : 0);
    return 0;
  }
  if (std::strcmp(name, "stream_half") == 0) {
    h->stream_half = value ? 1 : 0;
    return 0;
  }
  if (std::strcmp(name, "fused_resid") == 0) {
    h->fused_resid = value ? 1 : 0;
    return 0;
  }
  if (std::strcmp(name, "pdl") == 0) {
    h->lctx.use_pdl = value ? 1 : 0;   // programmatic dependent launch of the forward's kernel chain
    return 0;
  }
  if (std::strcmp(name, "dconv_mma") == 0) {
    h->dconv_mma = value ? 1 : 0;
    return 0;
  }
  if (std::strcmp(name, "l2_discard") == 0) {
    h->l2_discard = value ? 1 : 0;
    return 0;
  }
  if (std::strcmp(name, "precision") == 0) {
    if (value < 0 || value > 2) return fail(h, SEPTFA_E_INVALID, "precision must be 0 (auto), 1 (fast) or 2 (accurate)");
    h->precision = value;
    return 0;
  }
  if (std::strcmp(name, "host_chunks") == 0) {
    if (value < 0 || value > kHostChunksMax) return fail(h, SEPTFA_E_INVALID, "host_chunks must be 0..8");
    h->host_chunks = value;
    return 0;
  }
  return fail(h, SEPTFA_E_INVALID, std::string("unknown option ") + name);
}
int septfa_get_option(const septfa_handle* h, const char* name) {
  if (h && name && std::strcmp(name, "engine") == 0) return h->engine;
  if (h && name && std::strcmp(name, "profile") == 0) return h->profile;
  if (h && name && std::strcmp(name, "precision") == 0) return h->precision;
  return SEPTFA_E_INVALID;
}

int septfa_commit_weights(septfa_handle* h) {
  if (!h) return SEPTFA_E_INVALID;
  for (const auto& k : h->keys)
    if (!h->host.count(k.name)) return fail(h, SEPTFA_E_KEY, "missing key " + k.name);
  CUDA_TRY(h, cudaSetDevice(h->device));
  for (void* p : h->allocs) cudaFree(p);
  h->allocs.clear();
  h->blocks.assign(h->nblk, DevBlock{});
  const auto& c = h->cfg;

  // The two analysis windows must agree (they always do: both are hann buffers, model.py:383-385);
  // the STFT is then computed once instead of twice (model.py:408-409).
  if (T_(h, "spec_input.spec.window") != T_(h, "spec_output.window"))
    return fail(h, SEPTFA_E_INVALID, "spec_input.spec.window and spec_output.window differ: unsupported");
  if (upload(h, T_(h, "spec_output.window"), &h->win_fwd)) return SEPTFA_E_CUDA;
  if (upload(h, T_(h, "inv_spec.window"), &h->win_inv)) return SEPTFA_E_CUDA;
  {
    std::vector<float2> tw(512);
    make_twiddles(tw.data());
    if (upload(h, tw, &h->twiddle)) return SEPTFA_E_CUDA;
  }
  if (upload(h, T_(h, "TCN.LN.weight"), &h->ln_g) || upload(h, T_(h, "TCN.LN.bias"), &h->ln_b)) return SEPTFA_E_CUDA;

  for (int i = 0; i < h->nblk; ++i) {
    DevBlock& d = h->blocks[i];
    const std::string p = "TCN.TCN." + std::to_string(i);
    d.dil = (i % c.layer) % 4 + 1;  // model.py:285-293
    // conv1d 256 -> 256
    {
      const auto w = fold_wn(T_(h, p + ".conv1d.weight_g"), T_(h, p + ".conv1d.weight_v"), kC);
      std::vector<float> wt((size_t)kC * kC);
      for (int n = 0; n < kC; ++n)
        for (int k = 0; k < kC; ++k) wt[(size_t)k * kC + n] = (float)w[(size_t)n * kC + k];
      // tcgen05 engine: the affine (gamma, beta) of the norm that produces this block's input is folded into
      // the weights / bias, so the A operand is the plain standardised stream (x - mean) * rstd.
      const std::vector<float>* gin = nullptr; const std::vector<float>* bin = nullptr;
      if (i == 0) { gin = &T_(h, "TCN.LN.weight"); bin = &T_(h, "TCN.LN.bias"); }
      else if (c.apply_recursive_ln) {
        gin = &T_(h, "TCN.ln_second_modules." + std::to_string(i - 1) + ".weight");
        bin = &T_(h, "TCN.ln_second_modules." + std::to_string(i - 1) + ".bias");
      }
      std::vector<double> wf(w);
      std::vector<float> b1f(T_(h, p + ".conv1d.bias"));
      if (gin) {
        for (int n = 0; n < kC; ++n) {
          double acc = 0.0;
          for (int k = 0; k < kC; ++k) {
            acc += w[(size_t)n * kC + k] * (double)(*bin)[k];
            wf[(size_t)n * kC + k] = w[(size_t)n * kC + k] * (double)(*gin)[k];
          }
          b1f[n] = (float)((double)b1f[n] + acc);
        }
      }
      {
        std::vector<float> sb(4 * 128);
        for (int n = 0; n < kC; ++n) {
          double srow = 0.0;
          for (int k = 0; k < kC; ++k) srow += (double)__half2float(__float2half((float)wf[(size_t)n * kC + k]));   // the fp16 operand the tensor core sees
          sb[(n / 2) * 4 + (n & 1)] = (float)srow;
          sb[(n / 2) * 4 + 2 + (n & 1)] = b1f[n];
        }
        const float* sp = nullptr;
        if (upload(h, sb, &sp)) return SEPTFA_E_CUDA;
        d.sb1 = reinterpret_cast<const float4*>(sp);
      }
      {
        // TF32 operand image (gemm_conv1_pair.cu): weights rounded to nearest at 11 significant bits, 8 K-chunks of 32 floats,
        // each chunk = 256 rows x 128 B, K-major with the 128-byte swizzle (16-byte unit index XOR row % 8)
        auto tf32_rn = [](float v) { uint32_t b; std::memcpy(&b, &v, 4); b = (b + 0x1000u) & 0xFFFFE000u; std::memcpy(&v, &b, 4); return v; };
        std::vector<float> img((size_t)kC * kC, 0.f), sb(4 * 128);
        for (int n = 0; n < kC; ++n) {
          double srow = 0.0;
          for (int k = 0; k < kC; ++k) {
            const float v = tf32_rn((float)wf[(size_t)n * kC + k]);
            srow += (double)v;
            const int j = k >> 5, kk = k & 31;
            const size_t byte = (size_t)j * 256 * 128 + (size_t)(n >> 3) * 1024 + (size_t)(n & 7) * 128 + (size_t)(((kk >> 2) ^ (n & 7)) << 4) + (size_t)(kk & 3) * 4;
            img[byte / 4] = v;
          }
          sb[(n / 2) * 4 + (n & 1)] = (float)srow;
          sb[(n / 2) * 4 + 2 + (n & 1)] = b1f[n];
        }
        const float* sp = nullptr;
        if (upload(h, img, &d.w1_img32) || upload(h, sb, &sp)) return SEPTFA_E_CUDA;
        d.sb1_32 = reinterpret_cast<const float4*>(sp);
      }
      if (upload(h, pack_image(wf, kC, kC, 1, 256), &d.w1_img) || upload(h, pack_image(split_lo(wf), kC, kC, 1, 256), &d.w1_img_lo) ||
          upload(h, wt, &d.w1_t) ||
          upload(h, T_(h, p + ".conv1d.bias"), &d.b1) || upload(h, b1f, &d.b1f))
        return SEPTFA_E_CUDA;
      d.a1 = T_(h, p + ".nonlinearity1.weight")[0];
      if (upload(h, T_(h, p + ".reg1.weight"), &d.g1) || upload(h, T_(h, p + ".reg1.bias"), &d.be1)) return SEPTFA_E_CUDA;
    }
    // depthwise 256 -> 512, k3
    {
      const auto w = fold_wn(T_(h, p + ".dconv1d.weight_g"), T_(h, p + ".dconv1d.weight_v"), kH);
      const auto& b2 = T_(h, p + ".dconv1d.bias");
      const auto& g1v = T_(h, p + ".reg1.weight");
      const auto& be1v = T_(h, p + ".reg1.bias");
      std::vector<float4> w2b(kH), w2f(kH);
      std::vector<float> c2f(kH);
      for (int o = 0; o < kH; ++o) {
        w2b[o] = make_float4((float)w[o * 3], (float)w[o * 3 + 1], (float)w[o * 3 + 2], b2[o]);
        const double g = g1v[o / 2], be = be1v[o / 2];
        const double f0 = w[o * 3] * g, f1 = w[o * 3 + 1] * g, f2 = w[o * 3 + 2] * g;
        w2f[o] = make_float4((float)f0, (float)f1, (float)f2, (float)(f0 + f1 + f2));
        c2f[o] = (float)((double)b2[o] + be * (w[o * 3] + w[o * 3 + 1] + w[o * 3 + 2]));
      }
      if (upload(h, w2b, &d.w2b) || upload(h, w2f, &d.w2f) || upload(h, c2f, &d.c2f)) return SEPTFA_E_CUDA;
      d.a2 = T_(h, p + ".nonlinearity2.weight")[0];
      // tcgen05 producer (gemm_tc.cu, MODE 1): the same folded taps arranged for packed pairs. Lane chunk c8 of K-chunk j
      // produces outputs 64 j + 8 c8 + e; pair (gp, par) = outputs e = 4 gp + par and e + 2, i.e. the equal-parity outputs
      // of input channels 2 gp and 2 gp + 1. Tables [j][pair][c8]: A = {wx_a, wx_b, wy_a, wy_b}, B = {wz_a, wz_b, sw_a,
      // sw_b}, C = {c2f_a, c2f_b}. Zero padding is realised by substituting the input that normalises to zero,
      // mean - (beta / gamma) / rstd, so gamma must not vanish: |gamma| is clamped to 1e-20 (the folded tap w * gamma and
      // the substitute then still multiply to the exact -w * beta / rstd).
      {
        std::vector<float> tab(2560), bog(kC);
        auto gsafe = [&](int c) { const double g = g1v[c]; return std::fabs(g) < 1e-20 ? (g < 0 ? -1e-20 : 1e-20) : g; };
        for (int c = 0; c < kC; ++c) bog[c] = (float)((double)be1v[c] / gsafe(c));
        for (int j = 0; j < 8; ++j)
          for (int pr = 0; pr < 4; ++pr)
            for (int c8 = 0; c8 < 8; ++c8) {
              const int idx = (j * 4 + pr) * 8 + c8, gp = pr >> 1, par = pr & 1;
              const int oa = 64 * j + 8 * c8 + 4 * gp + par, ob = oa + 2;
              double f[2][3], sw[2], cf[2];
              const int oo[2] = {oa, ob};
              for (int e = 0; e < 2; ++e) {
                const int o = oo[e];
                const double g = gsafe(o / 2), be = be1v[o / 2];
                for (int k = 0; k < 3; ++k) f[e][k] = w[o * 3 + k] * g;
                sw[e] = f[e][0] + f[e][1] + f[e][2];
                cf[e] = (double)b2[o] + be * (w[o * 3] + w[o * 3 + 1] + w[o * 3 + 2]);
              }
              float* A = tab.data() + idx * 4;
              float* Bt = tab.data() + 1024 + idx * 4;
              float* Ct = tab.data() + 2048 + idx * 2;
              A[0] = (float)f[0][0]; A[1] = (float)f[1][0]; A[2] = (float)f[0][1]; A[3] = (float)f[1][1];
              Bt[0] = (float)f[0][2]; Bt[1] = (float)f[1][2]; Bt[2] = (float)sw[0]; Bt[3] = (float)sw[1];
              Ct[0] = (float)cf[0]; Ct[1] = (float)cf[1];
            }
        const float* tptr = nullptr;
        if (upload(h, tab, &tptr) || upload(h, bog, &d.bog)) return SEPTFA_E_CUDA;
        d.wtab = reinterpret_cast<const float4*>(tptr);
      }
      // dconv_mma2.cu: the depthwise conv as block-diagonal tensor-core GEMMs. Group gi = input channels 16 gi .. +15 ->
      // outputs 32 gi .. +31; per tap k a B operand [32 outputs][16 inputs] with B[n][n / 2] = fp16(w[o][k] * gamma1[o / 2])
      // and zeros elsewhere, split along the outputs into the halves the two CTAs of a pair hold: per rank [16 outputs][16
      // inputs] (fp16, K-major, no swizzle: core matrices of 8 rows x 16 B, the two K halves 256 B apart).
      // The kernel's affine uses the SAME rounded taps (sw = their sum, c2f = b2 + beta / gamma * sw), so the result is
      // an exact depthwise conv with the effective weights fp16(w gamma) / gamma.
      {
        std::vector<uint8_t> img2(kDconvTapBytes, 0);
        std::vector<float> swc(4 * 256), w16(3 * kH);
        bool ok = true;
        for (int cch = 0; cch < kC; ++cch) ok = ok && std::isfinite(g1v[cch]) && std::fabs(g1v[cch]) >= 1e-3f;
        for (int o = 0; o < kH; ++o) {
          double sw = 0.0;
          for (int k = 0; k < 3; ++k) {
            const float f = (float)(w[o * 3 + k] * (double)g1v[o / 2]);
            ok = ok && std::isfinite(f) && std::fabs(f) < 60000.f;
            const __half hq = __float2half(f);
            const float fq = __half2float(hq);
            w16[k * kH + o] = fq;
            sw += (double)fq;
            const int gi = o / 32, n = o % 32, kk = (o / 2) % 16;
            // pair layout: [rank = n / 16][group][tap][K half][16 outputs][8 inputs]
            const size_t byte2 = (size_t)(n / 16) * (kDconvTapBytes / 2) + (size_t)((gi * 3 + k) * 512) + (size_t)(kk / 8) * 256 +
                                 (size_t)(n % 16) * 16 + (size_t)(kk % 8) * 2;
            std::memcpy(img2.data() + byte2, &hq, 2);
          }
          const double bogv = ok ? (double)be1v[o / 2] / (double)g1v[o / 2] : 0.0;
          swc[(o / 2) * 4 + (o & 1)] = (float)sw;
          swc[(o / 2) * 4 + 2 + (o & 1)] = (float)((double)b2[o] + bogv * sw);
        }
        const float* sp = nullptr;
        if (upload(h, img2, &d.tap_img2) || upload(h, swc, &sp) || upload(h, w16, &d.w16)) return SEPTFA_E_CUDA;
        d.swc = reinterpret_cast<const float4*>(sp);
        d.mma_ok = ok;
      }
    }
    // res_out 512 -> 256 with GroupNorm reg2 folded in:  r = rstd2 * (W3g q - mu2 * s3) + c03
    {
      const auto w = fold_wn(T_(h, p + ".res_out.weight_g"), T_(h, p + ".res_out.weight_v"), kC);
      const auto& g2 = T_(h, p + ".reg2.weight");
      const auto& be2 = T_(h, p + ".reg2.bias");
      const auto& b3 = T_(h, p + ".res_out.bias");
      std::vector<double> wg((size_t)kC * kH);
      std::vector<float> wt((size_t)kH * kC), s3_tc(kC), s3_ref(kC), c03(kC);
      for (int n = 0; n < kC; ++n) {
        double s_tc = 0.0, s_ref = 0.0, c0 = (double)b3[n];
        for (int o = 0; o < kH; ++o) {
          const double v = w[(size_t)n * kH + o] * (double)g2[o];
          wg[(size_t)n * kH + o] = v;
          wt[(size_t)o * kC + n] = (float)v;
          s_tc += (double)__half2float(__float2half((float)v));  // matches the fp16 operand the tensor core sees
          s_ref += (double)(float)v;
          c0 += w[(size_t)n * kH + o] * (double)be2[o];
        }
        s3_tc[n] = (float)s_tc;
        s3_ref[n] = (float)s_ref;
        c03[n] = (float)c0;
      }
      if (upload(h, pack_image(wg, kC, kH, 1, 256), &d.w3_img) || upload(h, pack_image(split_lo(wg), kC, kH, 1, 256), &d.w3_img_lo) ||
          upload(h, wt, &d.w3_t) || upload(h, s3_tc, &d.s3_tc) ||
          upload(h, s3_ref, &d.s3_ref) || upload(h, c03, &d.c03))
        return SEPTFA_E_CUDA;
    }
    d.tf.enabled = c.tf_attention;
    if (c.tf_attention) {
      const std::string q = "TCN.time_freq_attnetion." + std::to_string(i);
      for (int k = 0; k < 3; ++k) {
        d.tf.wt1[k] = T_(h, q + ".conv1d_t_1.weight")[k];
        d.tf.wt2[k] = T_(h, q + ".conv1d_t_2.weight")[k];
        d.tf.wf1[k] = T_(h, q + ".conv1d_f_1.weight")[k];
        d.tf.wf2[k] = T_(h, q + ".conv1d_f_2.weight")[k];
      }
      d.tf.bt1 = T_(h, q + ".conv1d_t_1.bias")[0];
      d.tf.bt2 = T_(h, q + ".conv1d_t_2.bias")[0];
      d.tf.bf1 = T_(h, q + ".conv1d_f_1.bias")[0];
      d.tf.bf2 = T_(h, q + ".conv1d_f_2.bias")[0];
      d.tf.at = T_(h, q + ".prelu_t.weight")[0];
      d.tf.af = T_(h, q + ".prelu_f.weight")[0];
    }
    if (c.apply_recursive_ln) {
      const std::string a = "TCN.ln_first_modules." + std::to_string(i), b = "TCN.ln_second_modules." + std::to_string(i);
      if (upload(h, T_(h, a + ".weight"), &d.lf_g) || upload(h, T_(h, a + ".bias"), &d.lf_b) ||
          upload(h, T_(h, b + ".weight"), &d.ls_g) || upload(h, T_(h, b + ".bias"), &d.ls_b))
        return SEPTFA_E_CUDA;
    } else if (c.apply_residual_ln) {
      const std::string a = "TCN.ln_modules." + std::to_string(i);
      if (upload(h, T_(h, a + ".weight"), &d.lm_g) || upload(h, T_(h, a + ".bias"), &d.lm_b)) return SEPTFA_E_CUDA;
    }
  }
  // output layer 256 -> 514 (padded to 576 = 3 x 192)
  {
    h->out_a = T_(h, "TCN.output.0.weight")[0];
    auto w = fold_wn(T_(h, "TCN.output.2.weight_g"), T_(h, "TCN.output.2.weight_v"), kBins * 2);
    std::vector<float> wt((size_t)kC * kLogitStride, 0.f), bias(kLogitStride, 0.f);
    for (int n = 0; n < kBins * 2; ++n) bias[n] = T_(h, "TCN.output.2.bias")[n];
    int nvalid = kBins * 2;
    if (c.final_vad) {
      // VAD.common.conv1_1 (257 -> 4, k5) applied to the logits is linear in them, so its 2 x 20 per-frame partial
      // products  part[s][k][j] = sum_f w1[j][f][k] logit[s*257 + f]  are 40 more outputs of THIS contraction with the
      // composite weights W1 * Wo (and bias W1 * bo). They live in the padding columns kVadCol0 .. +39 of the 576-wide
      // logits rows: no extra pass over the logits (the former k_vad_partial: 118 us, LSU-bound), no extra GEMM tile.
      const auto w1 = fold_wn(T_(h, "vad.common.conv1_1.weight_g"), T_(h, "vad.common.conv1_1.weight_v"), 4);  // [4][257][5]
      nvalid = kVadCol0 + 40;
      w.resize((size_t)nvalid * kC, 0.0);
      for (int s2 = 0; s2 < 2; ++s2)
        for (int k = 0; k < 5; ++k)
          for (int j = 0; j < 4; ++j) {
            const int n = kVadCol0 + s2 * 20 + k * 4 + j;
            double bacc = 0.0;
            for (int f = 0; f < kBins; ++f) {
              const double w1v = w1[((size_t)j * kBins + f) * 5 + k];
              bacc += w1v * (double)bias[s2 * kBins + f];
              for (int kc = 0; kc < kC; ++kc) w[(size_t)n * kC + kc] += w1v * w[(size_t)(s2 * kBins + f) * kC + kc];
            }
            bias[n] = (float)bacc;
          }
    }
    const std::vector<double> w_lo = split_lo(w);   // low part of the 2-term fp16 split used by the tcgen05 output conv
    for (int n = 0; n < nvalid; ++n)
      for (int k = 0; k < kC; ++k) wt[(size_t)k * kLogitStride + n] = (float)w[(size_t)n * kC + k];
    if (upload(h, T_(h, "TCN.output.1.weight"), &h->out_g) || upload(h, T_(h, "TCN.output.1.bias"), &h->out_be) ||
        upload(h, pack_image(w, nvalid, kC, 3, 192), &h->out_img) || upload(h, pack_image(w_lo, nvalid, kC, 3, 192), &h->out_img_lo) ||
        upload(h, wt, &h->out_wt) ||
        upload(h, bias, &h->out_bias))
      return SEPTFA_E_CUDA;
  }
  if (c.final_vad) {
    const auto w2 = fold_wn(T_(h, "vad.output_layer_vad.weight_g"), T_(h, "vad.output_layer_vad.weight_v"), 1);  // [1][4][3]
    for (int j = 0; j < 4; ++j) {
      h->vad_b1[j] = T_(h, "vad.common.conv1_1.bias")[j];
      h->vad_g[j] = T_(h, "vad.common.BN_1.weight")[j];
      h->vad_be[j] = T_(h, "vad.common.BN_1.bias")[j];
      for (int k = 0; k < 3; ++k) h->vad_w2[j * 3 + k] = (float)w2[j * 3 + k];
    }
    h->vad_a = T_(h, "vad.common.relu_1.weight")[0];
    h->vad_b2 = T_(h, "vad.output_layer_vad.bias")[0];
  }
  if (c.activity_input_bool) {
    for (int i = 0; i < 9; ++i) h->act_k[i] = T_(h, "activity_input.weight")[i];
    h->act_b = T_(h, "activity_input.bias")[0];
    h->act_a = T_(h, "prelu.weight")[0];
  }
  h->all_mma_ok = true;
  for (const auto& d : h->blocks) h->all_mma_ok = h->all_mma_ok && d.mma_ok;
  h->committed = true;
  return 0;
}

size_t septfa_workspace_bytes(const septfa_handle* h, int B, int64_t L) {
  if (!h || B < 1 || L < 257) return 0;
  return carve(h, nullptr, B, L).total + 256;
}

int septfa_forward(septfa_handle* h, const float* x, int B, int64_t L, const septfa_infer_kw* kw, float* out_wav,
                   float* out_vad, void* est_stft, float* mask, float* spectrum, float* logits_out, void* workspace,
                   size_t workspace_bytes, void* stream) {
  if (int rc = check_forward_args(h, B, L)) return rc;
  if (!x || !out_wav || !workspace) return fail(h, SEPTFA_E_INVALID, "null x / out_wav / workspace");
  if (h->cfg.final_vad && !out_vad) return fail(h, SEPTFA_E_INVALID, "out_vad is required when final_vad is set");
  if (workspace_bytes < septfa_workspace_bytes(h, B, L)) return fail(h, SEPTFA_E_WORKSPACE, "workspace too small");
  CUDA_TRY(h, cudaSetDevice(h->device));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  void* base = reinterpret_cast<void*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255);
  const Workspace ws = carve(h, base, B, L);
  const int T = (int)septfa_num_frames(L);
  const int M = B * T;
  const auto& c = h->cfg;
  bind_ctx(&h->lctx);
  const ForwardPlan pl = plan_forward(*h, B, L, est_stft != nullptr || mask != nullptr || logits_out != nullptr);
  ctx().launches = 0;

  prof_mark(h, SEPTFA_PROF_FRONTEND, st);
  CUDA_TRY(h, cudaMemsetAsync(ws.zero_begin, 0, ws.zero_bytes, st));
  launch_frontend(x, B, L, T, h->win_fwd, h->twiddle, c.activity_input_bool, h->act_k, h->act_b, h->act_a, ws.S, ws.w,
                  ws.dcg, ws.st0, spectrum, st);   // (the optional spectrum export leaves from the front end's own rows)

  const int Mp = pl.Mp;
  if (pl.planes) {   // the halo slots of the plane layout must read as zeros
    uint8_t* pb = reinterpret_cast<uint8_t*>(ws.p);
    CUDA_TRY(h, cudaMemset2DAsync(pb, (size_t)Mp * 16, 0, (size_t)kPlaneHalo * 16, 32, st));
    CUDA_TRY(h, cudaMemset2DAsync(pb + (size_t)(M + kPlaneHalo) * 16, (size_t)Mp * 16, 0, (size_t)(Mp - M - kPlaneHalo) * 16, 32, st));
  }
  alignas(64) CUtensorMap wh_tmap;
  if (pl.conv1_rest == Conv1Kernel::tma && !make_stream_tmap(&wh_tmap, ws.wh, M))
    return fail(h, SEPTFA_E_CUDA, "cuTensorMapEncodeTiled failed for the fp16 stream");
  alignas(64) CUtensorMap w32_tmap;
  if (pl.conv1_rest == Conv1Kernel::pair && !make_stream_tmap(&w32_tmap, ws.w, M, 128, true))
    return fail(h, SEPTFA_E_CUDA, "cuTensorMapEncodeTiled failed for the fp32 stream");
  alignas(64) CUtensorMap racc_tmap;   // the pair kernel's epilogue stores racc with TMA tensor stores (boxes of 32 rows x 64 columns)
  if (pl.dconv == DconvKernel::mma2 && !make_stream_tmap(&racc_tmap, ws.racc, M, 32))
    return fail(h, SEPTFA_E_CUDA, "cuTensorMapEncodeTiled failed for racc");
  const double inv_n = 1.0 / ((double)kC * T);
  StreamNorm norm{ws.st0, h->ln_g, h->ln_b, 1e-8f, inv_n};  // TCN.LN, model.py:333
  for (int i = 0; i < h->nblk; ++i) {
    const DevBlock& d = h->blocks[i];
    Stat2* st_p = ws.st_blk + (size_t)(i * 4 + 0) * B;
    Stat2* st_q = ws.st_blk + (size_t)(i * 4 + 1) * B;
    Stat2* st_v = ws.st_blk + (size_t)(i * 4 + 2) * B;
    Stat2* st_w = ws.st_blk + (size_t)(i * 4 + 3) * B;
    double* colsum = ws.colsum + (size_t)i * B * kC;
    __half* p_planes = reinterpret_cast<__half*>(ws.p);

    prof_mark(h, SEPTFA_PROF_CONV1, st);
    const Conv1Params c1{ws.w, norm, M, T, B, d.b1, d.a1, d.w1_img, d.b1f, d.w1_t, ws.p, st_p, pl.half_io, pl.planes, Mp,
                         d.w1_img_lo, pl.split};
    switch (i == 0 ? pl.conv1_first : pl.conv1_rest) {
      case Conv1Kernel::ref: launch_ref_conv1(c1, st); break;
      case Conv1Kernel::tc_gemm: launch_tc_conv1(c1, st); break;
      case Conv1Kernel::persist: launch_conv1_persist(c1, st); break;
      case Conv1Kernel::pair:
        launch_conv1_pair(Conv1PairParams{&w32_tmap, norm, M, T, B, d.w1_img32, d.sb1_32, d.a1, p_planes, Mp, st_p}, st);
        break;
      case Conv1Kernel::tma:
        launch_conv1_tma(Conv1TmaParams{&wh_tmap, norm, M, T, B, d.w1_img, d.sb1, d.a1, p_planes, Mp, st_p}, st);
        break;
    }

    prof_mark(h, SEPTFA_PROF_DCONV, st);
    if (pl.dconv == DconvKernel::mma2) {
      launch_dconv_mma2(DconvMmaParams{p_planes, Mp, st_p, d.tap_img2, d.swc, d.w16, d.bog, d.a2, d.dil, M, T, B, d.w3_img,
                                       reinterpret_cast<__half*>(ws.racc), ws.rowsum, colsum, st_q, &racc_tmap, h->l2_discard},
                        st);
    } else {
      const DconvParams dc{ws.p, st_p, d.g1, d.be1, d.w2b, d.w2f, d.c2f, d.a2, d.dil, M, T, B, d.w3_img, d.w3_t, ws.racc,
                           ws.rowsum, colsum, st_q, pl.half_io, d.wtab, d.bog, d.w3_img_lo, pl.split};
      if (pl.dconv == DconvKernel::tc_gemm) launch_tc_dconv(dc, st); else launch_ref_dconv(dc, st);
    }

    const GateParams gp{st_q, (pl.dconv != DconvKernel::ref && !pl.split) ? d.s3_tc : d.s3_ref, d.c03, ws.rowsum, colsum, d.tf,
                        M, T, B, ws.ra, ws.rb, ws.gf, ws.gt, ws.mt};
    ResidParams rp{};
    rp.w = ws.w; rp.norm = norm; rp.racc = ws.racc; rp.racc_half = pl.half_io; rp.ra = ws.ra; rp.rb = ws.rb; rp.gf = ws.gf; rp.gt = ws.gt;
    rp.M = M; rp.T = T; rp.B = B; rp.mode = h->ln_mode; rp.st_v = st_v; rp.st_w = st_w; rp.discard = h->l2_discard;
    const bool in_half = pl.stream_half && i > 0, out_half = pl.stream_half && i + 1 < h->nblk;
    if (in_half) rp.w_half_in = ws.wh;
    if (out_half) rp.w_half_out = ws.wh;
    if (h->ln_mode == LN_RECURSIVE) { rp.g_a = d.lf_g; rp.b_a = d.lf_b; }        // model.py:347-348
    else if (h->ln_mode == LN_RESIDUAL) { rp.g_a = d.lm_g; rp.b_a = d.lm_b; }    // model.py:349-350
    if (const int clusters = pl.resid_clusters[in_half][out_half]) {
      prof_mark(h, SEPTFA_PROF_RESID, st);
      launch_resid_fused(rp, gp, clusters, st);
    } else {
      prof_mark(h, SEPTFA_PROF_GATE, st);
      launch_tf_gate(gp, st);
      prof_mark(h, SEPTFA_PROF_RESID, st);
      if (h->ln_mode != LN_NONE) launch_resid_stats(rp, st);
      launch_resid_apply(rp, st);
    }
    if (h->ln_mode == LN_RECURSIVE) norm = StreamNorm{st_w, d.ls_g, d.ls_b, 1e-5f, inv_n};   // output = ln_second(...)
    else norm = StreamNorm{nullptr, nullptr, nullptr, 0.f, inv_n};
  }
  // output layer: PReLU -> GroupNorm -> conv (model.py:322-325,357)
  prof_mark(h, SEPTFA_PROF_OUTCONV, st);
  launch_out_stats(ws.w, norm, h->out_a, M, T, ws.st_o, st);
  const OutConvParams oc{ws.w, norm, h->out_a, ws.st_o, h->out_g, h->out_be, M, T, B, h->out_bias, h->out_img, h->out_img_lo, h->out_wt, ws.logits};
  if (pl.tc_out) launch_tc_outconv(oc, st); else launch_ref_outconv(oc, st);

  prof_mark(h, SEPTFA_PROF_VAD, st);
  const bool use_kw = kw != nullptr && c.final_vad;  // `if inference_kw and self.final_vad`, model.py:444
  const float* gate = nullptr;
  if (c.final_vad) {
    VadParams vp{};
    vp.logits = ws.logits; vp.M = M; vp.T = T; vp.B = B;
    std::memcpy(vp.b1, h->vad_b1, sizeof(vp.b1)); vp.slope = h->vad_a;
    std::memcpy(vp.g, h->vad_g, sizeof(vp.g)); std::memcpy(vp.be, h->vad_be, sizeof(vp.be));
    std::memcpy(vp.w2, h->vad_w2, sizeof(vp.w2)); vp.b2 = h->vad_b2;
    vp.c4 = ws.c4; vp.prob = ws.prob; vp.smooth = ws.smooth;
    vp.thr = use_kw ? kw->threshold_activated_vad : 0.f;
    vp.do_smooth = use_kw ? 1 : 0;
    launch_vad(vp, st);
    if (use_kw && (kw->filter_signals_by_smo_vad || kw->filter_signals_by_unsmo_vad)) gate = ws.smooth;  // model.py:452-455
    const float* vsrc = (use_kw && kw->return_smoothed_vad) ? ws.smooth : ws.prob;                      // model.py:456-457
    CUDA_TRY(h, cudaMemcpyAsync(out_vad, vsrc, (size_t)M * 2 * sizeof(float), cudaMemcpyDeviceToDevice, st));
  }
  prof_mark(h, SEPTFA_PROF_ISTFT, st);
  if (pl.exports)
    launch_mask_istft_export(ws.S, ws.logits, gate, h->win_inv, h->twiddle, B, L, T, out_wav, reinterpret_cast<float2*>(est_stft),
                             mask, logits_out, st);
  else
    launch_mask_istft(ws.S, ws.logits, gate, h->win_inv, h->twiddle, B, L, T, out_wav, st);
  prof_mark(h, -1, st);
  h->last_launches = ctx().launches;
  CUDA_TRY(h, cudaGetLastError());
  return 0;
}

int septfa_profile_read(septfa_handle* h, double* ms, int* launches, int n, int reset) {
  if (!h || !ms || n < SEPTFA_PROF_NCAT) return SEPTFA_E_INVALID;
  CUDA_TRY(h, cudaSetDevice(h->device));
  if (h->ev_used > 0) {
    CUDA_TRY(h, cudaEventSynchronize(h->ev_pool[h->ev_used - 1]));
    for (int i = 0; i + 1 < h->ev_used; ++i) {
      const int cat = h->ev_cat[i];
      if (cat < 0) continue;
      float t = 0.f;
      CUDA_TRY(h, cudaEventElapsedTime(&t, h->ev_pool[i], h->ev_pool[i + 1]));
      h->prof_ms[cat] += t;
      h->prof_launches[cat] += 1;
    }
    h->ev_used = 0;
  }
  for (int i = 0; i < SEPTFA_PROF_NCAT; ++i) {
    ms[i] = h->prof_ms[i];
    if (launches) launches[i] = h->prof_launches[i];
    if (reset) { h->prof_ms[i] = 0; h->prof_launches[i] = 0; }
  }
  return 0;
}

int septfa_forward_host(septfa_handle* h, const float* x_host, int B, int64_t L, const septfa_infer_kw* kw,
                        float* out_wav_host, float* out_vad_host) {
  if (int rc = check_forward_args(h, B, L)) return rc;
  if (!x_host || !out_wav_host) return fail(h, SEPTFA_E_INVALID, "null host buffer");
  CUDA_TRY(h, cudaSetDevice(h->device));
  if (!h->hstream) {
    CUDA_TRY(h, cudaStreamCreateWithFlags(&h->hstream, cudaStreamNonBlocking));
    CUDA_TRY(h, cudaStreamCreateWithFlags(&h->hstream_in, cudaStreamNonBlocking));
    CUDA_TRY(h, cudaStreamCreateWithFlags(&h->hstream_out, cudaStreamNonBlocking));
    for (int i = 0; i < kHostChunksMax; ++i) {
      CUDA_TRY(h, cudaEventCreateWithFlags(&h->hev_in[i], cudaEventDisableTiming));
      CUDA_TRY(h, cudaEventCreateWithFlags(&h->hev_done[i], cudaEventDisableTiming));
    }
  }
  const int64_t T = septfa_num_frames(L);
  // Independent utterances: the batch is cut into chunks that alternate between two stream "lanes". Each lane
  // runs copy-in -> kernels -> copy-out in order on its own stream and workspace; the two lanes overlap each
  // other's copies with kernels and keep the SMs filled while one lane's (smaller) grids drain.
  // measured on B200, 256 x 4 s (tools/e2e_sweep.py): 1 chunk 8.9 ms, 2 chunks 7.5 ms, 4 chunks 8.5 ms, 8 chunks 12.7 ms
  int nchunk = h->host_chunks > 0 ? h->host_chunks : (B >= 64 ? 2 : 1);
  nchunk = std::min(std::min(nchunk, kHostChunksMax), B);
  const int Bc = (B + nchunk - 1) / nchunk;
  const size_t nx = (size_t)B * L * sizeof(float), nout = nx * 2, nvad = (size_t)B * 2 * T * sizeof(float);
  const size_t nws = septfa_workspace_bytes(h, Bc, L);
  auto grow = [&](float** dev, float** pin, size_t* cap, size_t need) -> cudaError_t {
    if (*cap >= need) return cudaSuccess;
    cudaFree(*dev); cudaFreeHost(*pin);
    *dev = nullptr; *pin = nullptr; *cap = 0;
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(dev), need);
    if (e != cudaSuccess) return e;
    e = cudaMallocHost(reinterpret_cast<void**>(pin), need);
    if (e == cudaSuccess) *cap = need;
    return e;
  };
  CUDA_TRY(h, grow(&h->hx_dev, &h->hx_pin, &h->hcap_x, nx));
  CUDA_TRY(h, grow(&h->hout_dev, &h->hout_pin, &h->hcap_out, nout));
  CUDA_TRY(h, grow(&h->hvad_dev, &h->hvad_pin, &h->hcap_vad, nvad));
  if (h->hcap_ws < nws) {
    cudaFree(h->hws); h->hws = nullptr; h->hcap_ws = 0;
    CUDA_TRY(h, cudaMalloc(&h->hws, nws));
    h->hcap_ws = nws;
  }
  if (nchunk > 1 && h->hcap_ws_b < nws) {
    cudaFree(h->hws_b); h->hws_b = nullptr; h->hcap_ws_b = 0;
    CUDA_TRY(h, cudaMalloc(&h->hws_b, nws));
    h->hcap_ws_b = nws;
  }
  // Page-locked caller buffers are copied directly; pageable ones go through the pinned staging buffers.
  auto is_pinned = [](const void* p) {
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeHost;
  };
  const bool pin_x = is_pinned(x_host), pin_out = is_pinned(out_wav_host);
  const bool want_vad = h->cfg.final_vad && out_vad_host != nullptr;
  const bool pin_vad = want_vad && is_pinned(out_vad_host);
  if (!pin_x) std::memcpy(h->hx_pin, x_host, nx);
  const float* xsrc = pin_x ? x_host : h->hx_pin;
  float* odst = pin_out ? out_wav_host : h->hout_pin;
  float* vdst = pin_vad ? out_vad_host : h->hvad_pin;
  int launches = 0;
  for (int c = 0; c < nchunk; ++c) {
    const int b0 = c * Bc, bn = std::min(Bc, B - b0);
    if (bn <= 0) break;
    const int lane = c & 1;
    cudaStream_t ls = lane ? h->hstream_in : h->hstream;
    void* lws = lane ? h->hws_b : h->hws;
    const size_t lcap = lane ? h->hcap_ws_b : h->hcap_ws;
    const size_t xo = (size_t)b0 * L, oo = (size_t)b0 * 2 * L, vo = (size_t)b0 * 2 * T;
    CUDA_TRY(h, cudaMemcpyAsync(h->hx_dev + xo, xsrc + xo, (size_t)bn * L * sizeof(float), cudaMemcpyHostToDevice, ls));
    if (int rc = septfa_forward(h, h->hx_dev + xo, bn, L, kw, h->hout_dev + oo, h->hvad_dev + vo, nullptr, nullptr, nullptr,
                                nullptr, lws, lcap, ls))
      return rc;
    launches += h->last_launches;
    CUDA_TRY(h, cudaMemcpyAsync(odst + oo, h->hout_dev + oo, (size_t)bn * 2 * L * sizeof(float), cudaMemcpyDeviceToHost, ls));
    if (want_vad)
      CUDA_TRY(h, cudaMemcpyAsync(vdst + vo, h->hvad_dev + vo, (size_t)bn * 2 * T * sizeof(float), cudaMemcpyDeviceToHost, ls));
  }
  h->last_launches = launches;
  CUDA_TRY(h, cudaStreamSynchronize(h->hstream));
  CUDA_TRY(h, cudaStreamSynchronize(h->hstream_in));
  if (!pin_out) std::memcpy(out_wav_host, h->hout_pin, nout);
  if (want_vad && !pin_vad) std::memcpy(out_vad_host, h->hvad_pin, nvad);
  return 0;
}

int septfa_forward_host_submit(septfa_handle* h, int slot, const float* x_host, int B, int64_t L, const septfa_infer_kw* kw,
                               float* out_wav_host, float* out_vad_host) {
  return septfa_forward_host_submit_fmt(h, slot, x_host, SEPTFA_FMT_F32, B, L, kw, out_wav_host, SEPTFA_FMT_F32, out_vad_host);
}

int septfa_forward_host_submit_fmt(septfa_handle* h, int slot, const void* x_host, int x_fmt, int B, int64_t L,
                                   const septfa_infer_kw* kw, void* out_wav_host, int out_fmt, float* out_vad_host) {
  if (int rc = check_forward_args(h, B, L)) return rc;
  if (x_fmt != SEPTFA_FMT_F32 && x_fmt != SEPTFA_FMT_PCM16) return fail(h, SEPTFA_E_INVALID, "x_fmt must be SEPTFA_FMT_F32 or SEPTFA_FMT_PCM16");
  if (out_fmt != SEPTFA_FMT_F32 && out_fmt != SEPTFA_FMT_F16) return fail(h, SEPTFA_E_INVALID, "out_fmt must be SEPTFA_FMT_F32 or SEPTFA_FMT_F16");
  if (slot < 0 || slot >= SEPTFA_HOST_SLOTS) return fail(h, SEPTFA_E_INVALID, "slot must be 0 .. SEPTFA_HOST_SLOTS - 1");
  if (!x_host || !out_wav_host) return fail(h, SEPTFA_E_INVALID, "null host buffer");
  auto& sl = h->slots[slot];
  if (sl.busy) return fail(h, SEPTFA_E_STATE, "slot has a batch in flight: call septfa_forward_host_wait first");
  CUDA_TRY(h, cudaSetDevice(h->device));
  const bool want_vad = h->cfg.final_vad && out_vad_host != nullptr;
  auto is_pinned = [](const void* p) {
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeHost;
  };
  if (!is_pinned(x_host) || !is_pinned(out_wav_host) || (want_vad && !is_pinned(out_vad_host)))
    return fail(h, SEPTFA_E_INVALID, "septfa_forward_host_submit needs page-locked host buffers");
  if (!sl.stream) {
    CUDA_TRY(h, cudaStreamCreateWithFlags(&sl.stream, cudaStreamNonBlocking));
    CUDA_TRY(h, cudaEventCreateWithFlags(&sl.ev_in, cudaEventDisableTiming));
    CUDA_TRY(h, cudaEventCreateWithFlags(&sl.ev_done, cudaEventDisableTiming));
  }
  if (!h->slot_compute) CUDA_TRY(h, cudaStreamCreateWithFlags(&h->slot_compute, cudaStreamNonBlocking));
  const int64_t T = septfa_num_frames(L);
  const size_t nx = (size_t)B * L * sizeof(float), nout = nx * 2, nvad = (size_t)B * 2 * T * sizeof(float);
  const size_t nws = septfa_workspace_bytes(h, B, L);
  const bool pcm = x_fmt == SEPTFA_FMT_PCM16, half_out = out_fmt == SEPTFA_FMT_F16;
  auto grow = [&](void** dev, size_t* cap, size_t need) -> cudaError_t {
    if (*cap >= need) return cudaSuccess;
    cudaFree(*dev); *dev = nullptr; *cap = 0;
    cudaError_t e = cudaMalloc(dev, need);
    if (e == cudaSuccess) *cap = need;
    return e;
  };
  CUDA_TRY(h, grow(reinterpret_cast<void**>(&sl.x), &sl.cap_x, nx));
  CUDA_TRY(h, grow(reinterpret_cast<void**>(&sl.out), &sl.cap_out, nout));
  CUDA_TRY(h, grow(reinterpret_cast<void**>(&sl.vad), &sl.cap_vad, nvad));
  CUDA_TRY(h, grow(&sl.ws, &sl.cap_ws, nws));
  if (pcm) {
    CUDA_TRY(h, grow(&sl.xraw, &sl.cap_xraw, nx / 2));
    CUDA_TRY(h, grow(reinterpret_cast<void**>(&sl.ext), &sl.cap_ext, (size_t)B * 2 * sizeof(unsigned)));
  }
  if (half_out) CUDA_TRY(h, grow(&sl.out16, &sl.cap_out16, nout / 2));
  // Copies run on the slot's own stream, the kernels of BOTH slots on one compute stream in submission order: a
  // batch's forward has the SMs to itself (two interleaved 78-kernel chains were 15 % slower than back to back) while
  // the other slot's copy-in and copy-out use the two copy engines underneath it.
  // 16-bit formats halve the PCIe bytes either way: PCM16 input is converted and min-max normalised on the device
  // (only_inference.py:69,81), fp16 output is the precision_save=16 cast of save_audio (utlis_inference.py:30-32).
  if (pcm) CUDA_TRY(h, cudaMemcpyAsync(sl.xraw, x_host, nx / 2, cudaMemcpyHostToDevice, sl.stream));
  else CUDA_TRY(h, cudaMemcpyAsync(sl.x, x_host, nx, cudaMemcpyHostToDevice, sl.stream));
  CUDA_TRY(h, cudaEventRecord(sl.ev_in, sl.stream));
  CUDA_TRY(h, cudaStreamWaitEvent(h->slot_compute, sl.ev_in, 0));
  int extra = 0;
  if (pcm) {
    bind_ctx(&h->lctx);
    launch_minmax_normalize_pcm16(reinterpret_cast<const int16_t*>(sl.xraw), B, L, nullptr, sl.ext, sl.x, h->slot_compute);
    extra += 3;
  }
  if (int rc = septfa_forward(h, sl.x, B, L, kw, sl.out, sl.vad, nullptr, nullptr, nullptr, nullptr, sl.ws, sl.cap_ws, h->slot_compute))
    return rc;
  if (half_out) {
    launch_to_half(sl.out, reinterpret_cast<__half*>(sl.out16), (int64_t)B * 2 * L, h->slot_compute);
    extra += 1;
  }
  h->last_launches += extra;
  CUDA_TRY(h, cudaEventRecord(sl.ev_done, h->slot_compute));
  CUDA_TRY(h, cudaStreamWaitEvent(sl.stream, sl.ev_done, 0));
  if (half_out) CUDA_TRY(h, cudaMemcpyAsync(out_wav_host, sl.out16, nout / 2, cudaMemcpyDeviceToHost, sl.stream));
  else CUDA_TRY(h, cudaMemcpyAsync(out_wav_host, sl.out, nout, cudaMemcpyDeviceToHost, sl.stream));
  if (want_vad) CUDA_TRY(h, cudaMemcpyAsync(out_vad_host, sl.vad, nvad, cudaMemcpyDeviceToHost, sl.stream));
  sl.busy = true;
  return 0;
}

int septfa_forward_host_wait(septfa_handle* h, int slot) {
  if (!h) return SEPTFA_E_INVALID;
  if (slot < 0 || slot >= SEPTFA_HOST_SLOTS) return fail(h, SEPTFA_E_INVALID, "slot must be 0 .. SEPTFA_HOST_SLOTS - 1");
  auto& sl = h->slots[slot];
  if (!sl.busy) return fail(h, SEPTFA_E_STATE, "slot has no batch in flight");
  CUDA_TRY(h, cudaSetDevice(h->device));
  sl.busy = false;
  CUDA_TRY(h, cudaStreamSynchronize(sl.stream));
  return 0;
}

int septfa_last_launch_count(const septfa_handle* h) { return h ? h->last_launches : 0; }

// ------------------------------------------------------------------------------------------ CUDA-graph replay
int septfa_graph_capture(septfa_handle* h, const float* x, int B, int64_t L, const septfa_infer_kw* kw, float* out_wav,
                         float* out_vad, void* workspace, size_t workspace_bytes, septfa_graph** out) {
  if (!out) return SEPTFA_E_INVALID;
  *out = nullptr;
  if (int rc = check_forward_args(h, B, L)) return rc;
  CUDA_TRY(h, cudaSetDevice(h->device));
  // one eager forward first: it fills the lazily initialised caches (occupancy queries) and validates the arguments
  cudaStream_t cs = nullptr;
  CUDA_TRY(h, cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
  const int saved_profile = h->profile, saved_pdl = h->lctx.use_pdl;
  h->profile = 0;
  int rc = septfa_forward(h, x, B, L, kw, out_wav, out_vad, nullptr, nullptr, nullptr, nullptr, workspace, workspace_bytes, cs);
  if (rc == 0 && cudaStreamSynchronize(cs) != cudaSuccess) rc = fail(h, SEPTFA_E_CUDA, "eager forward before the capture failed");
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  // programmatic dependent launches are captured as programmatic edges; if this driver refuses them inside a capture,
  // the chain is captured with plain stream order instead
  for (int attempt = 0; rc == 0 && attempt < 2 && exec == nullptr; ++attempt) {
    h->lctx.use_pdl = attempt == 0 ? saved_pdl : 0;
    if (cudaStreamBeginCapture(cs, cudaStreamCaptureModeRelaxed) != cudaSuccess) { rc = fail(h, SEPTFA_E_CUDA, "cudaStreamBeginCapture failed"); break; }
    const int frc = septfa_forward(h, x, B, L, kw, out_wav, out_vad, nullptr, nullptr, nullptr, nullptr, workspace, workspace_bytes, cs);
    const cudaError_t ce = cudaStreamEndCapture(cs, &graph);
    if (frc == 0 && ce == cudaSuccess && graph != nullptr && cudaGraphInstantiate(&exec, graph, 0) == cudaSuccess) break;
    cudaGetLastError();
    if (graph) { cudaGraphDestroy(graph); graph = nullptr; }
    exec = nullptr;
    if (attempt == 1) rc = fail(h, SEPTFA_E_CUDA, "the forward could not be captured into a CUDA graph");
  }
  h->profile = saved_profile;
  h->lctx.use_pdl = saved_pdl;
  cudaStreamDestroy(cs);
  if (rc != 0 || exec == nullptr) return rc != 0 ? rc : SEPTFA_E_CUDA;
  auto* g = new septfa_graph();
  g->h = h; g->graph = graph; g->exec = exec;
  size_t n = 0;
  cudaGraphGetNodes(graph, nullptr, &n);
  g->nodes = (int)n;
  g->kernels = h->last_launches;
  *out = g;
  return 0;
}

int septfa_graph_launch(septfa_graph* g, void* stream) {
  if (!g) return SEPTFA_E_INVALID;
  CUDA_TRY(g->h, cudaGraphLaunch(g->exec, reinterpret_cast<cudaStream_t>(stream)));
  g->h->last_launches = g->kernels;
  return 0;
}

int septfa_graph_num_nodes(const septfa_graph* g) { return g ? g->nodes : 0; }

void septfa_graph_destroy(septfa_graph* g) {
  if (!g) return;
  cudaGraphExecDestroy(g->exec);
  cudaGraphDestroy(g->graph);
  delete g;
}

// ------------------------------------------------------------------------------------------ online
int septfa_online_create(septfa_handle* h, int S, septfa_online** out) {
  return septfa_online_create_win(h, S, kWinLen, kHopLen, out);
}

int septfa_online_create_win(septfa_handle* h, int S, int window, int hop, septfa_online** out) {
  if (!h || !out || S < 1 || S > 32767) return fail(h, SEPTFA_E_INVALID, "bad arguments (1 <= S <= 32767 streams per online state)");
  *out = nullptr;
  if (int rc = check_geometry(h, window, hop)) { h->last_launches = 0; return rc; }
  if (!h->committed) return fail(h, SEPTFA_E_STATE, "weights not committed");
  CUDA_TRY(h, cudaSetDevice(h->device));
  auto* o = new septfa_online();
  o->h = h;
  o->S = S;
  o->win = window;
  o->hop = hop;
  const size_t tb = (size_t)S * 2 * (window - hop) * sizeof(float);
  if (cudaMalloc(reinterpret_cast<void**>(&o->tail[0]), tb) != cudaSuccess ||
      cudaMalloc(reinterpret_cast<void**>(&o->tail[1]), tb) != cudaSuccess ||
      cudaMalloc(reinterpret_cast<void**>(&o->acc), (size_t)S * 4 * sizeof(double)) != cudaSuccess) {
    cudaFree(o->tail[0]); cudaFree(o->tail[1]); cudaFree(o->acc);
    delete o;
    return fail(h, SEPTFA_E_CUDA, "online state allocation failed");
  }
  *out = o;
  return 0;
}

void septfa_online_destroy(septfa_online* o) {
  if (!o) return;
  cudaSetDevice(o->h->device);
  cudaFree(o->tail[0]); cudaFree(o->tail[1]); cudaFree(o->acc);
  delete o;
}

int septfa_online_reset(septfa_online* o, void*) {
  if (!o) return SEPTFA_E_INVALID;
  o->hops = 0; o->tail_len = 0; o->cur = 0;
  return 0;
}

int septfa_online_hops_done(const septfa_online* o) { return o ? o->hops : 0; }

size_t septfa_online_workspace_bytes(const septfa_online* o) {
  if (!o) return 0;
  const size_t pred = ((size_t)o->S * 2 * o->win * sizeof(float) + 255) & ~(size_t)255;
  const size_t vad = ((size_t)o->S * 2 * septfa_num_frames(o->win) * sizeof(float) + 255) & ~(size_t)255;
  return pred + vad + septfa_workspace_bytes(o->h, o->S, o->win) + 256;
}

int septfa_online_step(septfa_online* o, const float* win, const septfa_infer_kw* kw, float* emitted, int32_t* perm,
                       void* workspace, size_t workspace_bytes, void* stream) {
  if (!o || !win || !emitted || !perm || !workspace) return SEPTFA_E_INVALID;
  septfa_handle* h = o->h;
  if (workspace_bytes < septfa_online_workspace_bytes(o)) return fail(h, SEPTFA_E_WORKSPACE, "online workspace too small");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255);
  const size_t pred_b = ((size_t)o->S * 2 * o->win * sizeof(float) + 255) & ~(size_t)255;
  const size_t vad_b = ((size_t)o->S * 2 * septfa_num_frames(o->win) * sizeof(float) + 255) & ~(size_t)255;
  float* pred = reinterpret_cast<float*>(base);
  float* vad = reinterpret_cast<float*>(base + pred_b);
  void* fws = base + pred_b + vad_b;
  // pred_separation, _, _ = self.model(truncated_signal_mix, inference_kw)   online_class_unknown_targets.py:84
  if (int rc = septfa_forward(h, win, o->S, o->win, kw, pred, vad, nullptr, nullptr, nullptr, nullptr, fws,
                              workspace_bytes - pred_b - vad_b - 256, st))
    return rc;
  int launches = h->last_launches;
  bind_ctx(&h->lctx);
  ctx().launches = 0;
  const int64_t Lw = o->win;
  const int hop = o->hop, tail_cap = o->win - o->hop;
  if (o->hops == 0) {
    // indx == 0: online_signal = pred[..., -hop:] (not yet reordered) is what the overlap is compared to (:85-88)
    launch_pit(pred + (Lw - 2 * hop), 2 * Lw, Lw, pred + (Lw - hop), 2 * Lw, Lw, o->S, hop, o->acc, perm, st);
  } else {
    const int n = o->tail_len;  // min(emitted so far, W - H)
    launch_pit(pred + (Lw - hop - n), 2 * Lw, Lw, o->tail[o->cur], 2 * (int64_t)tail_cap, tail_cap, o->S, n, o->acc,
               perm, st);
  }
  // pred = reorder_source_mse(pred, perm); online_signal = cat(online_signal, pred[..., -hop:])   (:93-94)
  launch_online_emit(pred, Lw, perm, o->S, hop, tail_cap, o->tail[o->cur], o->tail_len, o->tail[o->cur ^ 1], emitted, st);
  o->cur ^= 1;
  o->tail_len = std::min(o->tail_len + hop, tail_cap);
  o->hops += 1;
  h->last_launches = launches + ctx().launches;
  CUDA_TRY(h, cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------ live sessions
}  // extern "C"

namespace {

struct LiveWorkspace {
  int32_t* slots;   // [n] device copy of the push's slot list
  float* win;       // [n, W]
  float* pred;      // [n, 2, W]
  float* vad;       // [n, 2, T(W)]
  float* u;         // [n, H] the resampled hops (sessions at a rate other than 16000)
  float* y;         // [n, 2, H] the emitted 16 kHz hops (sessions at an output rate other than 16000)
  void* fws;        // the forward's workspace
  size_t fws_bytes;
  size_t total;
};

LiveWorkspace live_carve(const septfa_live* lv, uintptr_t base, int n) {
  auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
  const int W = lv->g.win;
  LiveWorkspace w{};
  size_t off = 0;
  w.slots = reinterpret_cast<int32_t*>(base + off); off += al((size_t)n * sizeof(int32_t));
  w.win = reinterpret_cast<float*>(base + off);     off += al((size_t)n * W * sizeof(float));
  w.pred = reinterpret_cast<float*>(base + off);    off += al((size_t)n * 2 * W * sizeof(float));
  w.vad = reinterpret_cast<float*>(base + off);     off += al((size_t)n * 2 * septfa_num_frames(W) * sizeof(float));
  if (lv->rate != kResampleRate) { w.u = reinterpret_cast<float*>(base + off); off += al((size_t)n * lv->g.hop * sizeof(float)); }
  if (lv->out_rate != kResampleRate) {
    w.y = reinterpret_cast<float*>(base + off);
    off += al((size_t)n * 2 * lv->g.hop * sizeof(float));
  }
  w.fws = reinterpret_cast<void*>(base + off);
  w.fws_bytes = septfa_workspace_bytes(lv->h, n, W);
  w.total = off + w.fws_bytes;
  return w;
}

// A slot list comes from the host: it is checked in full before anything is launched, since a bad entry would index the
// per-slot state out of bounds on the device and a duplicate would make two CTAs race on one slot.
int check_live_slots(septfa_live* lv, const int32_t* slots, int n) {
  septfa_handle* h = lv->h;
  if (!slots) return fail(h, SEPTFA_E_INVALID, "null slot list");
  if (n < 1 || n > lv->capacity)
    return fail(h, SEPTFA_E_INVALID, "n = " + std::to_string(n) + ": a slot list holds 1 .. capacity (" +
                                         std::to_string(lv->capacity) + ") slots");
  std::vector<uint8_t> seen(lv->capacity, 0);
  for (int i = 0; i < n; ++i) {
    const int32_t s = slots[i];
    if (s < 0 || s >= lv->capacity)
      return fail(h, SEPTFA_E_INVALID, "slot " + std::to_string(s) + " (entry " + std::to_string(i) + ") out of range 0 .. " +
                                           std::to_string(lv->capacity - 1));
    if (seen[s]) return fail(h, SEPTFA_E_INVALID, "slot " + std::to_string(s) + " listed twice (entry " + std::to_string(i) + ")");
    seen[s] = 1;
  }
  return 0;
}

}  // namespace

extern "C" {

int septfa_live_create(septfa_handle* h, int capacity, septfa_live** out) {
  return septfa_live_create_win(h, capacity, kWinLen, kHopLen, out);
}

int septfa_live_create_win(septfa_handle* h, int capacity, int window, int hop, septfa_live** out) {
  return septfa_live_create_rate(h, capacity, window, hop, kResampleRate, out);
}

int septfa_live_create_rate(septfa_handle* h, int capacity, int window, int hop, int rate, septfa_live** out) {
  return septfa_live_create_rates(h, capacity, window, hop, rate, kResampleRate, out);
}

int septfa_live_create_rates(septfa_handle* h, int capacity, int window, int hop, int rate, int out_rate, septfa_live** out) {
  if (!h || !out || capacity < 1 || capacity > 32767)
    return fail(h, SEPTFA_E_INVALID, "bad arguments (1 <= capacity <= 32767 slots per live session)");
  *out = nullptr;
  if (int rc = check_geometry(h, window, hop)) { h->last_launches = 0; return rc; }
  ResamplePlan pl{};
  if (int rc = check_rate(h, rate, kToModel, &pl)) { h->last_launches = 0; return rc; }
  if (hop % pl.nw) {   // a push must carry a whole number of native samples
    h->last_launches = 0;
    return fail(h, SEPTFA_E_INVALID, "rate " + std::to_string(rate) + ", hop " + std::to_string(hop) +
                                         ": the hop must be a multiple of " + std::to_string(pl.nw) + " samples at this rate");
  }
  const int in_hop = (int)((int64_t)hop * pl.orig / pl.nw);
  if (pl.hist > in_hop) {
    h->last_launches = 0;
    return fail(h, SEPTFA_E_INVALID, "rate " + std::to_string(rate) + ", hop " + std::to_string(hop) +
                                         ": the resampler's history exceeds one hop");
  }
  ResamplePlan opl{};
  if (int rc = check_rate(h, out_rate, kFromModel, &opl)) { h->last_launches = 0; return rc; }
  if (hop % opl.orig) {   // a push must return a whole number of output samples
    h->last_launches = 0;
    return fail(h, SEPTFA_E_INVALID, "out rate " + std::to_string(out_rate) + ", hop " + std::to_string(hop) +
                                         ": the hop must be a multiple of " + std::to_string(opl.orig) +
                                         " samples at this output rate");
  }
  if (opl.hist > hop) {
    h->last_launches = 0;
    return fail(h, SEPTFA_E_INVALID, "out rate " + std::to_string(out_rate) + ", hop " + std::to_string(hop) +
                                         ": the output resampler's history exceeds one hop");
  }
  if (!h->committed) return fail(h, SEPTFA_E_STATE, "weights not committed");
  CUDA_TRY(h, cudaSetDevice(h->device));
  ResampleBank bank{}, out_bank{};
  if (rate != kResampleRate)
    if (int rc = get_bank(h, rate, kToModel, nullptr, &bank)) return rc;
  if (out_rate != kResampleRate)
    if (int rc = get_bank(h, out_rate, kFromModel, nullptr, &out_bank)) return rc;
  auto* lv = new septfa_live();
  lv->h = h;
  lv->capacity = capacity;
  lv->rate = rate;
  lv->in_hop = in_hop;
  lv->bank = bank;
  lv->out_rate = out_rate;
  lv->out_hop = (int)((int64_t)hop * opl.nw / opl.orig);
  lv->out_bank = out_bank;
  const int first = (window - hop + 255) / 256;   // the first window frame whose centre 256 j lies in [W - H, W)
  lv->g = LiveGeom{window, hop, first, (window + 255) / 256 - first};
  const size_t ring_b = (size_t)(window - hop) * sizeof(float);
  const size_t hist_b = (size_t)capacity * 2 * std::max(bank.hist, 1) * sizeof(float);
  const size_t hist_out_b = (size_t)capacity * 4 * std::max(out_bank.hist, 1) * sizeof(float);
  if (cudaMalloc(reinterpret_cast<void**>(&lv->hops_done), (size_t)capacity * sizeof(int32_t)) != cudaSuccess ||
      cudaMalloc(reinterpret_cast<void**>(&lv->in_ring), (size_t)capacity * ring_b) != cudaSuccess ||
      cudaMalloc(reinterpret_cast<void**>(&lv->tail_ring), (size_t)capacity * 2 * ring_b) != cudaSuccess ||
      (rate != kResampleRate && cudaMalloc(reinterpret_cast<void**>(&lv->hist), hist_b) != cudaSuccess) ||
      (out_rate != kResampleRate && cudaMalloc(reinterpret_cast<void**>(&lv->hist_out), hist_out_b) != cudaSuccess) ||
      cudaMemset(lv->hops_done, 0, (size_t)capacity * sizeof(int32_t)) != cudaSuccess) {
    cudaFree(lv->hops_done); cudaFree(lv->in_ring); cudaFree(lv->tail_ring); cudaFree(lv->hist); cudaFree(lv->hist_out);
    delete lv;
    return fail(h, SEPTFA_E_CUDA, "live session allocation failed");
  }
  *out = lv;
  return 0;
}

void septfa_live_destroy(septfa_live* lv) {
  if (!lv) return;
  cudaSetDevice(lv->h->device);
  cudaFree(lv->hops_done); cudaFree(lv->in_ring); cudaFree(lv->tail_ring); cudaFree(lv->hist); cudaFree(lv->hist_out);
  delete lv;
}

int septfa_live_input_hop(const septfa_live* lv, int* delay) {
  if (!lv) return SEPTFA_E_INVALID;
  if (delay) *delay = lv->rate == kResampleRate ? 0 : lv->bank.delay;
  return lv->in_hop;
}

int septfa_live_output_hop(const septfa_live* lv, int* delay) {
  if (!lv) return SEPTFA_E_INVALID;
  if (delay) *delay = lv->out_rate == kResampleRate ? 0 : lv->out_bank.delay;
  return lv->out_hop;
}

size_t septfa_live_workspace_bytes(const septfa_live* lv, int n) {
  if (!lv || n < 1 || n > lv->capacity) return 0;
  return live_carve(lv, 0, n).total + 256;
}

int septfa_live_vad_frames(const septfa_live* lv, int* first_frame) {
  if (!lv) return SEPTFA_E_INVALID;
  if (first_frame) *first_frame = lv->g.vad_frame0;
  return lv->g.vad_frames;
}

int septfa_live_release(septfa_live* lv, const int32_t* slots_host, int n, void* stream) {
  if (!lv) return SEPTFA_E_INVALID;
  septfa_handle* h = lv->h;
  if (int rc = check_live_slots(lv, slots_host, n)) return rc;
  CUDA_TRY(h, cudaSetDevice(h->device));
  bind_ctx(&h->lctx);
  launch_live_release(slots_host, n, lv->hops_done, reinterpret_cast<cudaStream_t>(stream));
  CUDA_TRY(h, cudaGetLastError());
  return 0;
}

int septfa_live_push(septfa_live* lv, const int32_t* slots_host, int n, const float* hops, const septfa_infer_kw* kw,
                     float* out, float* out_vad, int32_t* perm, void* workspace, size_t workspace_bytes, void* stream) {
  if (!lv) return SEPTFA_E_INVALID;
  septfa_handle* h = lv->h;
  // every check comes before the first launch: a push that fails leaves every slot as it was
  h->last_launches = 0;
  if (int rc = check_live_slots(lv, slots_host, n)) return rc;
  if (!hops || !out || !perm || !workspace) return fail(h, SEPTFA_E_INVALID, "null hops / out / perm / workspace");
  if (out_vad && !h->cfg.final_vad) return fail(h, SEPTFA_E_INVALID, "out_vad needs a model with a VAD head (final_vad)");
  if (!h->committed) return fail(h, SEPTFA_E_STATE, "weights not committed");
  if (workspace_bytes < septfa_live_workspace_bytes(lv, n)) return fail(h, SEPTFA_E_WORKSPACE, "live workspace too small");
  CUDA_TRY(h, cudaSetDevice(h->device));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const LiveWorkspace ws = live_carve(lv, (reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255, n);
  CUDA_TRY(h, cudaMemcpyAsync(ws.slots, slots_host, (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  bind_ctx(&h->lctx);
  ctx().launches = 0;
  if (lv->rate != kResampleRate) {
    launch_live_resample(ws.slots, n, lv->hops_done, lv->hist, hops, ws.u, lv->bank, lv->g.hop, lv->in_hop, st);
    hops = ws.u;
  }
  launch_live_window(ws.slots, n, lv->hops_done, lv->in_ring, hops, ws.win, lv->g, st);
  const int before = ctx().launches;
  if (int rc = septfa_forward(h, ws.win, n, lv->g.win, kw, ws.pred, ws.vad, nullptr, nullptr, nullptr, nullptr, ws.fws,
                              ws.fws_bytes, st))
    return rc;
  const int launches = before + h->last_launches;
  bind_ctx(&h->lctx);
  ctx().launches = 0;
  const bool out_resample = lv->out_rate != kResampleRate;
  launch_live_pit_emit(ws.slots, n, lv->hops_done, ws.pred, ws.vad, (int)septfa_num_frames(lv->g.win), lv->tail_ring,
                       out_resample ? ws.y : out, out_vad, perm, lv->g, st);
  if (out_resample)
    launch_live_out_resample(ws.slots, n, lv->hops_done, lv->hist_out, ws.y, out, lv->out_bank, lv->g.hop, lv->out_hop, st);
  h->last_launches = launches + ctx().launches;
  CUDA_TRY(h, cudaGetLastError());
  return 0;
}

int septfa_pit_l1(septfa_handle* h, const float* a, const float* b, int S, int64_t n, int32_t* perm, double* pw_sums,
                  void* stream) {
  if (!h || !a || !b || !perm || S < 1 || S > 65535 || n < 1) return SEPTFA_E_INVALID;
  CUDA_TRY(h, cudaSetDevice(h->device));
  if (h->pit_cap < S) {
    cudaFree(h->pit_acc); h->pit_acc = nullptr; h->pit_cap = 0;
    CUDA_TRY(h, cudaMalloc(reinterpret_cast<void**>(&h->pit_acc), (size_t)S * 4 * sizeof(double)));
    h->pit_cap = S;
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  bind_ctx(&h->lctx);
  launch_pit(a, 2 * n, n, b, 2 * n, n, S, n, h->pit_acc, perm, st);
  if (pw_sums) CUDA_TRY(h, cudaMemcpyAsync(pw_sums, h->pit_acc, (size_t)S * 4 * sizeof(double), cudaMemcpyDeviceToDevice, st));
  CUDA_TRY(h, cudaGetLastError());
  return 0;
}

int septfa_minmax_normalize(septfa_handle* h, const float* x, int B, int64_t L, const int64_t* lengths, float* out, void* stream) {
  if (!h || !x || !out || B < 1 || B > 65535 || L < 1) return fail(h, SEPTFA_E_INVALID, "bad arguments (1 <= B <= 65535)");
  CUDA_TRY(h, cudaSetDevice(h->device));
  if (h->norm_cap < B) {
    cudaFree(h->norm_ext); h->norm_ext = nullptr; h->norm_cap = 0;
    CUDA_TRY(h, cudaMalloc(reinterpret_cast<void**>(&h->norm_ext), (size_t)B * 2 * sizeof(unsigned)));
    h->norm_cap = B;
  }
  bind_ctx(&h->lctx);
  launch_minmax_normalize(x, B, L, lengths, h->norm_ext, out, reinterpret_cast<cudaStream_t>(stream));
  h->last_launches = 3;
  CUDA_TRY(h, cudaGetLastError());
  return 0;
}

int septfa_resample_geometry(int rate, int* delay, int* hop_multiple) {
  ResamplePlan pl{};
  if (int rc = check_rate(nullptr, rate, kToModel, &pl)) return rc;
  if (delay) *delay = pl.delay;
  if (hop_multiple) *hop_multiple = pl.nw;
  return 0;
}

int septfa_resample_to_geometry(int rate, int* delay, int* hop_multiple) {
  ResamplePlan pl{};
  if (int rc = check_rate(nullptr, rate, kFromModel, &pl)) return rc;
  if (delay) *delay = pl.delay;
  if (hop_multiple) *hop_multiple = pl.orig;   // the 16 kHz side is the source here
  return 0;
}

}  // extern "C"

namespace {

// The batch resampler of both directions: x [B, L] (float32, or int16 PCM to 16 kHz) -> out [B, ceil(nw L / orig)].
int resample_batch(septfa_handle* h, const void* x, int x_fmt, int B, int64_t L, int rate, ResampleDir dir, float* out,
                   void* stream) {
  if (!h) return SEPTFA_E_INVALID;
  h->last_launches = 0;
  if (!x || !out || B < 1 || B > 65535 || L < 1) return fail(h, SEPTFA_E_INVALID, "bad arguments (1 <= B <= 65535, L >= 1)");
  if (x_fmt != SEPTFA_FMT_F32 && x_fmt != SEPTFA_FMT_PCM16)
    return fail(h, SEPTFA_E_INVALID, "x_fmt must be SEPTFA_FMT_F32 or SEPTFA_FMT_PCM16");
  ResamplePlan pl{};
  if (int rc = check_rate(h, rate, dir, &pl)) return rc;
  CUDA_TRY(h, cudaSetDevice(h->device));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int64_t Lo = resample_out_len(pl, L);
  if (rate == kResampleRate && x_fmt == SEPTFA_FMT_F32) {
    CUDA_TRY(h, cudaMemcpyAsync(out, x, (size_t)B * L * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return 0;
  }
  ResampleBank bk{};
  if (int rc = get_bank(h, rate, dir, st, &bk)) return rc;
  bind_ctx(&h->lctx);
  ctx().launches = 0;
  launch_resample(x, x_fmt == SEPTFA_FMT_PCM16, B, L, Lo, out, bk, st);
  h->last_launches = ctx().launches;
  CUDA_TRY(h, cudaGetLastError());
  return 0;
}

}  // namespace

extern "C" {

int septfa_resample(septfa_handle* h, const void* x, int x_fmt, int B, int64_t L, int rate, float* out, void* stream) {
  return resample_batch(h, x, x_fmt, B, L, rate, kToModel, out, stream);
}

int septfa_resample_to(septfa_handle* h, const float* y, int B, int64_t L, int rate, float* out, void* stream) {
  return resample_batch(h, y, SEPTFA_FMT_F32, B, L, rate, kFromModel, out, stream);
}

int septfa_sisdr(const float* preds, const float* target, int64_t rows, int64_t n, int zero_mean, float* out_db, double* scratch,
                 void* stream) {
  if (!preds || !target || !out_db || !scratch || rows < 1 || rows > 65535 || n < 1) return SEPTFA_E_INVALID;
  bind_ctx(nullptr);   // no handle: the process-default launch context
  launch_sisdr(preds, target, rows, n, zero_mean, scratch, out_db, reinterpret_cast<cudaStream_t>(stream));
  return cudaGetLastError() == cudaSuccess ? 0 : SEPTFA_E_CUDA;
}

}  // extern "C"
