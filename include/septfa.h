/*
 * septfa.h - C ABI of libseptfa.so: the B200 (sm_100a) Sep-TFAnet-VAD inference forward pass.
 *
 * This is the drop-in boundary for ONE path of the reference (BaekMS/Sep-TFAnet-VAD):
 *   - SeparationModel.__init__ / load_state_dict / forward      model/model.py:360-461
 *   - OnlineSaving.calc_online (one hop of the sliding window)  model/online_class_unknown_targets.py:72-105
 *   - PITLossWrapper('pw_pt', L1) + reorder_source_mse          model/pit_wrapper.py:149-177,261-312; model/combined_loss.py:63-78
 *
 * The reference boundary is a Python nn.Module (there is no FFI in the reference); the entry
 * points below are what a ctypes binding of that module needs: plain pointers and sizes, no
 * torch types. Conventions: every call returns 0 on success or a negative SEPTFA_E_* code and
 * never throws; septfa_last_error() gives the message. All device pointers are caller-owned
 * and must live on the handle's device. Calls are stream-ordered on `stream` (a cudaStream_t
 * passed as void*; NULL = legacy default stream) and do not synchronise the host, except the
 * *_host variants which return after their result is in host memory. One handle per device;
 * a handle is not thread-safe.
 *
 * Device tensor layouts (float32 unless noted) mirror the torch tensors of the reference:
 *   x        [B, L]                 mixture waveforms                     forward(x)          model.py:402
 *   out_wav  [B, 2, L]              separated waveforms                   out_separation      model.py:460
 *   out_vad  [B, 2, T]              VAD probabilities, or the smoothed {0,1} decisions when
 *                                   kw->return_smoothed_vad (reference shape [B,2,1,T])      model.py:424-457
 *   est_stft [B, 2, 257, T] float2  estimated STFTs (complex64), nullable  estimated_stfts    model.py:437,453
 *   mask     [B, 2, 257, T]         post-sigmoid masks, nullable           mask_per_speaker   model.py:429
 *   spectrum [B, 257, T]            gated dB spectrum, nullable            self.spectrum      model.py:412-419
 *   logits   [B, 514, T]            pre-sigmoid masks, nullable            self.masks_b       model.py:421
 * with T = 1 + L / 256 (n_fft 512, hop 256, centre/reflect padding; L >= 257).
 */
#ifndef SEPTFA_H_
#define SEPTFA_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SEPTFA_OK 0
#define SEPTFA_E_INVALID (-1)     /* bad argument / unsupported configuration */
#define SEPTFA_E_CUDA (-2)        /* CUDA runtime error */
#define SEPTFA_E_STATE (-3)       /* call order (weights not committed, ...) */
#define SEPTFA_E_KEY (-4)         /* unknown / missing / mis-sized state_dict key */
#define SEPTFA_E_WORKSPACE (-5)   /* workspace too small */

typedef struct septfa_handle septfa_handle;
typedef struct septfa_online septfa_online;

/* arch.args of config_with_vad.json / config_without_vad.json (config_with_vad.json:7-28),
 * consumed by SeparationModel.__init__ (model/model.py:362-391). Booleans are 0/1. */
typedef struct septfa_config {
  int32_t n_fft_bins;                 /* "n_fftBins": only 512 */
  int32_t bn_dim;                     /* "BN_dim": only 256 (= n_fftBins/2, model.py:377-380) */
  int32_t h_dim;                      /* "H_dim": only 512 */
  int32_t layer;                      /* "layer" (blocks per stack, dilation cycle) */
  int32_t stack;                      /* "stack" */
  int32_t num_spk;                    /* "num_spk": only 2 */
  int32_t skip;                       /* must be 0 */
  int32_t dilated;                    /* must be 1 */
  int32_t causal;                     /* "casual" (sic): must be 0 */
  int32_t weight_norm;                /* must be 1 */
  int32_t final_vad;                  /* VAD head present */
  int32_t final_vad_masked_speakers;  /* must be 0 */
  int32_t noisy_phase;                /* model.py:430-439 (both branches equal S*mask numerically) */
  int32_t activity_input_bool;        /* model.py:414-419 */
  int32_t tf_attention;               /* model.py:344-345 */
  int32_t apply_recursive_ln;         /* model.py:347-348 */
  int32_t apply_residual_ln;          /* model.py:349-350 */
} septfa_config;

/* inference_kw of forward (model/model.py:444-457; only_inference.py:102-108).
 * Pass NULL for the reference's empty dict (no gating, raw probabilities). */
typedef struct septfa_infer_kw {
  int32_t length_smoothing_filter;      /* accepted and ignored, like the reference (weights are overwritten with [1,0,1]) */
  float threshold_activated_vad;
  int32_t filter_signals_by_smo_vad;
  int32_t filter_signals_by_unsmo_vad;  /* also gates with the *smoothed* decisions (model.py:454-455) */
  int32_t return_smoothed_vad;
} septfa_infer_kw;

/* Engines for the dense contractions (1x1 convs): a bit mask of the contractions that run on the
 * plain fp32 CUDA-core kernels instead of the tcgen05 tensor cores (bring-up / numerics cross-check):
 * bit 0 = conv1d (256->256), bit 1 = dconv+res_out (512->256), bit 2 = output conv (256->514). */
#define SEPTFA_ENGINE_TCGEN05_F16 0 /* all on tcgen05: fp16 operands, fp32 TMEM accumulators (default) */
#define SEPTFA_ENGINE_FP32_SIMT 7   /* all on fp32 CUDA cores */

int septfa_create(septfa_handle** out, const septfa_config* cfg, int device);
void septfa_destroy(septfa_handle* h);
const char* septfa_last_error(const septfa_handle* h); /* h may be NULL: last create() error */
const char* septfa_version(void);

/* Weights: one call per reference state_dict entry, by its reference key
 * (e.g. "TCN.TCN.3.conv1d.weight_v"), raw float32 host data in torch's contiguous layout.
 * weight_norm folding (w = g*v/||v||) and tensor-core packing happen in septfa_commit_weights,
 * which fails with SEPTFA_E_KEY if any key the configuration requires is missing - the same
 * contract as load_state_dict(strict=True) (only_inference.py:57-60). */
int septfa_set_tensor(septfa_handle* h, const char* key, const float* host_data, int64_t numel);
int septfa_commit_weights(septfa_handle* h);
/* Number of keys the configuration expects, and the i-th key (for strict checking on the host side). */
int septfa_num_keys(const septfa_handle* h);
const char* septfa_key_name(const septfa_handle* h, int i);
int64_t septfa_key_numel(const septfa_handle* h, int i);

/* name = "engine" (SEPTFA_ENGINE_*), "profile" (0/1), "host_chunks" (0 = automatic, 1..8: number of
 * batch chunks septfa_forward_host pipelines over its two stream lanes); kernel-selection switches for
 * cross-checks (default 1): "fused_resid" (cluster-resident gate + residual kernel), "conv1_persist"
 * (persistent warp-specialised conv1 kernel), "pdl" (programmatic dependent launch of the kernel chain),
 * "dconv_mma" (tensor-core depthwise + res_out kernel on CTA pairs, cta_group::2, weights resident),
 * "conv1_pair" (TF32 CTA-pair conv1 fed by TMA from the fp32 stream; blocks 1 .. n-1 of the recursive-LN wiring;
 * 2 = at any batch size), "l2_discard" (the hand-off buffers inside a block are dropped from the L2 once they have been read);
 * "stream_half" (default 0): opt-in mode that stores the residual stream between blocks as fp16 - 11 % faster, but the
 * stream's rounding accumulates over all blocks (VAD probabilities within 2e-3 of the reference instead of 1e-3).
 * Any other name is refused with SEPTFA_E_INVALID ("unknown option"), among them the retired switches that selected a
 * kernel slower on every measured workload (the single-CTA depthwise kernel and its bring-up variants, the streamed-weight
 * form of the persistent conv1 kernel). */
/* "precision": arithmetic of the two block contractions (conv1d 256->256, res_out 512->256) on the tensor cores.
 *   SEPTFA_PRECISION_FAST      fp16 operands, one tcgen05 pass, fp16 storage of the tensors between them
 *   SEPTFA_PRECISION_ACCURATE  2-term fp16 split of both operands (three passes, fp32-accurate), fp32 storage
 *   SEPTFA_PRECISION_AUTO      (default) ACCURATE for apply_residual_ln (config_without_vad: the residual stream is
 *                              never re-normalised and accumulates the rounding of all blocks), FAST otherwise */
#define SEPTFA_PRECISION_AUTO 0
#define SEPTFA_PRECISION_FAST 1
#define SEPTFA_PRECISION_ACCURATE 2
int septfa_set_option(septfa_handle* h, const char* name, int value);
int septfa_get_option(const septfa_handle* h, const char* name);

int64_t septfa_num_frames(int64_t L); /* T = 1 + L/256 */
size_t septfa_workspace_bytes(const septfa_handle* h, int B, int64_t L);

/* SeparationModel.forward (model/model.py:402-461). Nullable outputs are skipped. */
int septfa_forward(septfa_handle* h, const float* x, int B, int64_t L, const septfa_infer_kw* kw,
                   float* out_wav, float* out_vad, void* est_stft, float* mask, float* spectrum,
                   float* logits, void* workspace, size_t workspace_bytes, void* stream);

/* Same, from/to HOST buffers: copies x host->device, runs forward, copies out_wav/out_vad back and
 * waits for completion. Page-locked caller buffers are used directly, pageable ones go through
 * pinned staging owned by the handle. The batch is processed in chunks so that copies overlap the
 * kernels (utterances are independent). This is the call a caller without device memory of its
 * own makes (only_inference.py:90-91 semantics). */
int septfa_forward_host(septfa_handle* h, const float* x_host, int B, int64_t L, const septfa_infer_kw* kw,
                        float* out_wav_host, float* out_vad_host);

/* Batch streams (only_inference.py's loop over files, model/model.py:402 per batch): the same from/to HOST forward,
 * split into an asynchronous submit and a wait so that successive batches overlap - while batch n computes, the
 * results of batch n-1 travel device->host and the input of batch n+1 host->device (copy engines and SMs all busy).
 * SEPTFA_HOST_SLOTS independent slots (0 .. 3), each with its own copy stream, device buffers and workspace (all slots
 * share one compute stream: a batch's forward has the SMs to itself). THREE slots in rotation keep the pipeline full: with
 * two, the copy-in of batch i + 1 queues behind the copy-out of batch i - 1 on the same slot and the compute stream idles
 * ~0.4 ms per 256 x 4 s step. A slot holds one batch in
 * flight: submit(slot) -> wait(slot) -> submit(slot) ... The host buffers must be page-locked (cudaHostAlloc /
 * cudaHostRegister / torch pin_memory) and stay valid and untouched until wait(slot) returns. */
#define SEPTFA_HOST_SLOTS 4
int septfa_forward_host_submit(septfa_handle* h, int slot, const float* x_host, int B, int64_t L, const septfa_infer_kw* kw,
                               float* out_wav_host, float* out_vad_host);
int septfa_forward_host_wait(septfa_handle* h, int slot);

/* The same submit with 16-bit sample formats on the host side, which halves the PCIe bytes in either direction:
 *   x_fmt   SEPTFA_FMT_F32   float32 waveforms, already normalised (what forward() takes)
 *           SEPTFA_FMT_PCM16 int16 PCM exactly as scipy.io.wavfile.read returns it (only_inference.py:68); the device then
 *                            does only_inference.py:69,81: astype(float32) and the min-max normalisation to [-0.9, 0.9],
 *                            bit-identical to the reference's numpy expression, before the forward
 *   out_fmt SEPTFA_FMT_F32   float32 waveforms
 *           SEPTFA_FMT_F16   IEEE half, round to nearest: the `-ps 16` format of save_audio (Our_utils/utlis_inference.py:30-32)
 * x_host: B*L elements of x_fmt; out_wav_host: B*2*L elements of out_fmt; out_vad_host: float32 as above. */
#define SEPTFA_FMT_F32 0
#define SEPTFA_FMT_PCM16 1
#define SEPTFA_FMT_F16 2
int septfa_forward_host_submit_fmt(septfa_handle* h, int slot, const void* x_host, int x_fmt, int B, int64_t L,
                                   const septfa_infer_kw* kw, void* out_wav_host, int out_fmt, float* out_vad_host);

/* ---- small-request serving: the forward as a CUDA graph (SURVEY.md section 8(f) rank 4) ---------------------------
 * A forward of one short mixture is ~80 kernels of a few microseconds each: launch-bound (0.9 ms for one 4 s mixture).
 * septfa_graph_capture records septfa_forward for one (B, L, kw) on the caller's STATIC device buffers (x, out_wav,
 * out_vad, workspace: same pointers at every replay) into an executable CUDA graph; septfa_graph_launch replays it on a
 * stream (the caller refreshes x before, reads out_wav / out_vad after, stream-ordered). One graph per shape bucket.
 * The optional exports (est_stft / mask / spectrum / logits) are not part of the graph. */
typedef struct septfa_graph septfa_graph;
int septfa_graph_capture(septfa_handle* h, const float* x, int B, int64_t L, const septfa_infer_kw* kw, float* out_wav,
                         float* out_vad, void* workspace, size_t workspace_bytes, septfa_graph** out);
int septfa_graph_launch(septfa_graph* g, void* stream);
int septfa_graph_num_nodes(const septfa_graph* g);
void septfa_graph_destroy(septfa_graph* g);

/* Number of GPU kernels launched by the last forward / online step / live push on this handle (0 after a refused push
 * or a create refused for its geometry). */
int septfa_last_launch_count(const septfa_handle* h);

/* Per-kernel-class device timing. With option "profile" = 1, forward records CUDA events on its
 * launch stream around each class of kernels; septfa_profile_read waits for them and returns the
 * accumulated milliseconds and interval counts per class (arrays of SEPTFA_PROF_NCAT). */
#define SEPTFA_PROF_FRONTEND 0 /* memset + STFT/dB + activity gate (+ spectrum export) */
#define SEPTFA_PROF_CONV1 1    /* tcgen05 GEMM 256->256 with GroupNorm prologue, PReLU/stats epilogue */
#define SEPTFA_PROF_DCONV 2    /* tcgen05 GEMM 512->256 with depthwise-conv prologue */
#define SEPTFA_PROF_GATE 3     /* TF-attention gates */
#define SEPTFA_PROF_RESID 4    /* post-block GroupNorm residual kernels */
#define SEPTFA_PROF_OUTCONV 5  /* output statistics + tcgen05 GEMM 256->514 */
#define SEPTFA_PROF_VAD 6      /* VAD head + smoothing */
#define SEPTFA_PROF_ISTFT 7    /* mask + inverse STFT overlap-add + the optional est / mask / logits exports */
#define SEPTFA_PROF_EXPORT 8   /* reads 0: the exports are written by the ISTFT class's kernel */
#define SEPTFA_PROF_NCAT 9
int septfa_profile_read(septfa_handle* h, double* ms, int* launches, int n, int reset);

/* ---- online mode: OnlineSaving.calc_online, one hop for S independent streams -------------
 * An online state has a window of W samples and a hop of H samples (OnlineSaving's max_len and
 * save_sec times fs); septfa_online_create is septfa_online_create_win with W = 48000, H = 16000.
 * Accepted: 256 <= H, 2 H <= W <= 160000, W and H multiples of 16 (1 ms); anything else is
 * refused with SEPTFA_E_INVALID before anything is allocated.
 * State kept on the device per stream: the last <= W - H samples of already-emitted
 * (permutation-fixed) signal. Each step takes the current windows win[S, W], runs forward, picks
 * per stream the speaker permutation that minimises the L1 distance between the window's overlap
 * with the emitted signal (PITLossWrapper pw_pt + L1Loss, n_src = 2, ties -> identity; at the
 * first step the window's [W - 2H, W - H) against its own [W - H, W)), reorders, and emits the
 * last hop: emitted[S, 2, H], perm[S, 2] (int32). */
int septfa_online_create(septfa_handle* h, int S, septfa_online** out);
int septfa_online_create_win(septfa_handle* h, int S, int window, int hop, septfa_online** out);
void septfa_online_destroy(septfa_online* st);
int septfa_online_reset(septfa_online* st, void* stream);
size_t septfa_online_workspace_bytes(const septfa_online* st);
int septfa_online_step(septfa_online* st, const float* win, const septfa_infer_kw* kw, float* emitted,
                       int32_t* perm, void* workspace, size_t workspace_bytes, void* stream);
int septfa_online_hops_done(const septfa_online* st);

/* ---- live streaming sessions: OnlineSaving for streams that start and end independently ---------------------------
 * A session has `capacity` slots (1 .. 32767); each slot hosts one stream at a time. Every stream of a session has a
 * window of W samples and a hop of H samples, fixed by septfa_live_create_win (septfa_live_create: W = 48000,
 * H = SEPTFA_LIVE_HOP = 16000). Accepted: 256 <= H, 2 H <= W <= 160000, W and H multiples of 16 (1 ms); W - H need not
 * be a multiple of H. Anything else is refused with SEPTFA_E_INVALID before anything is allocated.
 * A stream is a sequence of pushes of exactly one hop each (H float32 samples, already normalised by the caller). Push
 * k (0-based) of a stream runs the forward on the window concat(the stream's last W - H samples, zeros before its first
 * sample; the new hop) - the stream left-padded with W - H zeros, model/online_class_known_targets.py:92-93 - and returns
 *   out  [2, H]               separated audio for the stream's samples [H k, H (k + 1)): the window's last H samples,
 *                             speakers permuted;
 *   perm [2] (int32)          the permutation: the L1 PIT of online_class_unknown_targets.py:84-94 between the window's
 *                             [W - H - o, W - H) and the last o = min(H k, W - H) emitted samples (ties -> identity);
 *                             at k = 0 the window's [W - 2H, W - H) is compared with its own [W - H, W), like the
 *                             reference's first window;
 *   vad  [2, F] (nullable)    out_vad of the window (probabilities, or the smoothed decisions with
 *                             kw->return_smoothed_vad), the window frames j0 .. j0 + F - 1 whose centres 256 j lie in
 *                             [W - H, W): j0 = ceil((W - H) / 256), F = ceil(W / 256) - j0 (septfa_live_vad_frames),
 *                             speakers in the emitted order. Frame j is centred on stream sample H k - (W - H) + 256 j.
 *                             When 256 divides H and W - H, F = H / 256 and the frames of consecutive hops tile one
 *                             grid; otherwise consecutive grids are offset (at the default, 16000 = 62.5 x 256: by half
 *                             a frame; j0 = 125, F = 63). Needs a model with a VAD head.
 * So the concatenated out of a stream of N pushes equals OnlineSaving.calc_online (max_len = W / 16000, save_sec =
 * H / 16000) on that stream alone, left-padded with W - H zeros. septfa_live_release ends the streams in the listed
 * slots; the next push into such a slot starts a new stream at k = 0 and reads nothing of the old one.
 * Slot lists are host arrays of n distinct slots, 1 <= n <= capacity; a bad list (slot out of range, a slot twice, n out
 * of range) is refused with SEPTFA_E_INVALID before anything is launched. A push that returns an error leaves every slot
 * unchanged. Per slot the session keeps on the device a hop counter, the last W - H input samples and the last W - H
 * emitted samples of both speakers (12 (W - H) + 4 bytes: ~384 KB at the default). Pushes and releases are
 * stream-ordered and do not synchronise the host; issue all calls of a session on one stream. hops: device [n, Hn] (Hn = H
 * at 16 kHz, see septfa_live_create_rate);
 * out: device [n, 2, H]; out_vad: device [n, 2, F]; perm: device int32 [n, 2]; the workspace is sized by
 * septfa_live_workspace_bytes for pushes of up to n slots. */
#define SEPTFA_LIVE_HOP 16000
#define SEPTFA_LIVE_FRAMES_PER_HOP 63
typedef struct septfa_live septfa_live;
int septfa_live_create(septfa_handle* h, int capacity, septfa_live** out);
int septfa_live_create_win(septfa_handle* h, int capacity, int window, int hop, septfa_live** out);
/* A session whose streams arrive at `rate` Hz (septfa_resample_geometry's rates; septfa_live_create_win is this with
 * rate 16000). Push k of a stream carries Hn = H rate / 16000 native samples (septfa_live_input_hop); the hop H must be a
 * multiple of the rate's hop_multiple. The session resamples each stream on the device, carrying the history from push
 * to push, and then serves the 16 kHz stream u = concat(D zeros, septfa_resample(stream)) exactly as a 16 kHz session
 * would: push k returns u[H k, H (k + 1)), its permutation and VAD frames. D (0 at 16000) is the delay of the streaming
 * resampler: the outputs of a push before (k + 1) H - D need no native sample after the hop. So the output lags the
 * input by D extra samples (6 .. 12 at the rates in the table of septfa_resample_geometry); a caller aligning output with
 * input shifts by D. Per slot the session keeps 2 x (at most 2 width + orig) more floats; a new stream reads none of
 * them. At 16000 nothing is added and a push launches what it launched before. */
int septfa_live_create_rate(septfa_handle* h, int capacity, int window, int hop, int rate, septfa_live** out);
/* A session whose streams arrive at `rate` Hz and whose separated audio is returned at `out_rate` Hz (both in
 * septfa_resample_geometry's range and independent of each other; septfa_live_create_rate is this with out_rate 16000).
 * Let y_s be the 16 kHz stream of emitted channel s: the concatenated out of a 16 kHz-output session, after the PIT
 * reordering. Push k returns out [n, 2, Ho], Ho = H out_rate / 16000 (septfa_live_output_hop):
 *   out[s] = z_s[k Ho, (k + 1) Ho),   z_s = concat(D_out zeros, septfa_resample_to(y_s, out_rate)),
 * bit for bit. D_out (0 at 16000) is the delay of the streaming output resampler in output samples: the outputs of a push
 * before (k + 1) Ho - D_out need no 16 kHz sample after the hop (6 at 8 kHz, 18 at 48 kHz, 16 at 44.1 kHz; see
 * septfa_resample_to_geometry). The hop must also be a multiple of the output rate's hop_multiple. perm and out_vad stay
 * on the 16 kHz frame grid, unchanged. Per slot the session keeps 4 x (the output resampler's history) more floats
 * (4 x 12 at 48 kHz, 4 x 24 at 8 kHz); a new stream reads none of them. At out_rate 16000 nothing is added and a push launches what it launched
 * before; otherwise one more kernel runs after the emit. A refused create (bad rate, out rate, hop or geometry) returns
 * SEPTFA_E_INVALID before anything is allocated and sets the launch count to 0. */
int septfa_live_create_rates(septfa_handle* h, int capacity, int window, int hop, int rate, int out_rate, septfa_live** out);
/* Hn, the native samples per push; *delay (nullable) receives D. */
int septfa_live_input_hop(const septfa_live* lv, int* delay);
/* Ho, the output samples per push and channel; *delay (nullable) receives D_out. */
int septfa_live_output_hop(const septfa_live* lv, int* delay);
void septfa_live_destroy(septfa_live* lv);
/* F, the VAD frames per push; *first_frame (nullable) receives j0. */
int septfa_live_vad_frames(const septfa_live* lv, int* first_frame);
size_t septfa_live_workspace_bytes(const septfa_live* lv, int n);
int septfa_live_release(septfa_live* lv, const int32_t* slots_host, int n, void* stream);
int septfa_live_push(septfa_live* lv, const int32_t* slots_host, int n, const float* hops, const septfa_infer_kw* kw,
                     float* out, float* out_vad, int32_t* perm, void* workspace, size_t workspace_bytes, void* stream);

/* Stand-alone PIT for 2 sources (model/pit_wrapper.py:149-177,261-312): a[S,2,n], b[S,2,n] ->
 * perm[S,2] (int32), decided per stream; pw_sums (nullable, device double [S,4]) receives the
 * pairwise L1 sums sum_n|a_i - b_j| at [s][i*2+j]. */
int septfa_pit_l1(septfa_handle* h, const float* a, const float* b, int S, int64_t n, int32_t* perm, double* pw_sums,
                  void* stream);

/* Pre-processing of only_inference.py:81, batched on the device: per utterance
 *   out = 1.8 * (x - min(x)) / (max(x) - min(x)) - 0.9        (float32, the reference's operation order: bit-identical
 * to numpy; a constant signal gives NaN like the reference). x, out: device [B, L]; lengths (nullable, device int64 [B]):
 * valid samples per utterance for ragged batches - extrema over the valid part, zeros written behind it. */
int septfa_minmax_normalize(septfa_handle* h, const float* x, int B, int64_t L, const int64_t* lengths, float* out, void* stream);

/* Resampling to 16 kHz: torchaudio.functional.resample(x, rate, 16000) with its defaults (sinc_interp_hann,
 * lowpass_filter_width 6, rolloff 0.99), what read_mixture applies through transforms.Resample (only_inference.py:68-79).
 * Accepted rates: integers in [8000, 192000] Hz; anything else is refused with SEPTFA_E_INVALID. With g = gcd(rate,
 * 16000), orig = rate / g, new = 16000 / g, output m = b new + p is the fp32 FMA chain over the taps of phase p of a
 * polyphase bank computed in double on the host and stored as fp32, keeping only the taps whose scaled time |t| < 6
 * (torchaudio's taps beyond are ~1e-20 or smaller): within ~4e-7 of float64 torchaudio on inputs in [-0.9, 0.9].
 * septfa_resample_geometry needs no handle and no device: *delay (nullable) receives D, the delay in 16 kHz samples of
 * a streaming resampler fed in hops (septfa_live_create_rate), and *hop_multiple (nullable) receives `new`, which a live
 * hop must be a multiple of. D is 12 at 8000 Hz, 8 at 11025 and 12000 Hz and 6 at 22050 .. 192000 Hz. */
int septfa_resample_geometry(int rate, int* delay, int* hop_multiple);
/* x: device [B, L] at `rate` Hz, x_fmt SEPTFA_FMT_F32 (float32) or SEPTFA_FMT_PCM16 (int16 PCM, converted as
 * astype(float32), only_inference.py:69: no scaling); out: device float32 [B, ceil(16000 L / rate)]. Rate 16000 is the
 * identity. The first call at a rate builds its bank, uploads it and waits for the upload; later calls at that rate are
 * stream-ordered and do not synchronise the host. */
int septfa_resample(septfa_handle* h, const void* x, int x_fmt, int B, int64_t L, int rate, float* out, void* stream);

/* Resampling the model's 16 kHz output to `rate`: torchaudio.functional.resample(y, 16000, rate) with the same defaults
 * and the same bank construction with source and destination swapped (orig = 16000 / g, new = rate / g), within ~1e-6
 * of float64 torchaudio. Accepted rates are those of septfa_resample, refused the same way.
 * septfa_resample_to_geometry needs no handle and no device: *delay (nullable) receives D_out, the delay in output
 * samples of a streaming output resampler (septfa_live_create_rates), and *hop_multiple (nullable) receives 16000 / g,
 * which a live hop must be a multiple of. */
int septfa_resample_to_geometry(int rate, int* delay, int* hop_multiple);
/* y: device float32 [B, L] at 16 kHz; out: device float32 [B, ceil(rate L / 16000)]. Rate 16000 copies. The bank cache,
 * the first-call upload and the stream ordering are those of septfa_resample. */
int septfa_resample_to(septfa_handle* h, const float* y, int B, int64_t L, int rate, float* out, void* stream);

/* calc_sisdr (model/combined_loss.py:16-56): SI-SDR in dB of `rows` pairs preds[rows, n] / target[rows, n] (device,
 * float32, contiguous) in one pass; out_db device [rows]; scratch: device, rows * 5 doubles; rows <= 65535. Runs on the
 * current device (no handle). The online drivers use it for the online-vs-offline quality report of test.py:223-269. */
int septfa_sisdr(const float* preds, const float* target, int64_t rows, int64_t n, int zero_mean, float* out_db, double* scratch,
                 void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SEPTFA_H_ */
