// Persistent, warp-specialised tcgen05 kernel for the second half of a TCN block (model/model.py:136/142,144), on CTA pairs:
//   q = PReLU(depthwise dilated k3 conv(GN1(p))),  racc = (W3 diag(g2)) q,  statistics of q, row / column sums of racc
// with BOTH contractions on the tensor cores. The depthwise convolution is block-diagonal (output channel o reads input
// channel o/2), so for a group of 16 input channels and one tap k it is a tiny GEMM
//   D1[frames x 32 outputs] += P_k[frames x 16] * B_k[16 x 32],   P_k = the p tile shifted by (k-1)*dilation frames,
// whose A operand needs no data movement at all: p is stored by conv1 as per-K-group planes [32][rows][8 channels]
// (16 bytes per frame and plane), one TMA bulk copy brings a plane's 136 frames (tile + halo) into shared memory already
// in the canonical no-swizzle K-major core-matrix layout (8 frames x 16 B), and a shift by s frames is the same buffer
// addressed 16*s bytes further on. GroupNorm reg1 is folded into the taps (w' = w * gamma, fp16) and into a per-row affine
//   x = rstd * conv + (c2f - rstd * mean * sw),   q = PReLU(x)      (sw = sum of the fp16 taps, c2f = b2 + beta / gamma * sw)
// applied to the fp32 accumulator on its way from tensor memory to the fp16 A operand of the res_out GEMM, which takes it
// from tensor memory: q never touches shared memory. That is 9 SASS instructions per PAIR of q values (FFMA2 pipe) instead
// of ~34 for the CUDA-core depthwise producer of gemm_tc.cu (MODE 1), which bounded that kernel at 20 % of the tensor
// roofline.
// Zero padding of the NORMALISED signal (the reference pads h1, not p): the tensor-core convolution reads whatever
// neighbours the shifted view holds; the <= 2*dil rows per utterance whose tap falls outside are corrected exactly,
//   x_true = x_mma - w'_k * (rstd * (p_wrong - mean) + beta / gamma),
// with the same fp16 weight and fp16 input the tensor core multiplied.
//
// The CTAs run as PAIRS (clusters of two on one TPC) and every MMA is a tcgen05.mma.cta_group::2 of M = 256 (128 frames
// per CTA) issued by the pair's leader; the B operand of such an MMA is split along N between the two CTAs, so each CTA
// needs only HALF of the res_out weight image (128 of its 256 output rows: 128 KB) and half of every tap matrix (24 KB) -
// and those fit in shared memory for the whole persistent kernel. The per-tile traffic into an SM is its own 68 KB of p.
// (A single-CTA form has to re-stream the 256 KB image for every 128-frame tile, which bounds it at one SM's TMA ingress:
// ~20 B/clk, 1.95 k cycles per 64-channel chunk against 0.6 k cycles of MMA work.)
// Roles per CTA (16 warps):
//   warp 0        p loader   : 4 bulk copies (K-group planes) per 32-channel chunk, ring of 4
//   warp 1        static loader (prologue), then EDGE warp: the exact zero-padding corrections of the <= 8 rows of a tile whose
//                 tap falls outside their utterance, as a small table per p stage
//   warp 2        res_out MMA issuer (leader CTA): per chunk 4 MMAs (M256 N256 K16, A from TMEM) into D2; multicast commits
//   warp 3        leader: depthwise mini-MMA issuer, per chunk 6 MMAs (3 taps x 2 groups, M256 N32 K16) into the D1 ring, as far
//                 ahead as the ring allows; peer: relay ("my p slab / my weights have landed" -> the leader's barriers)
//   warps 4-11    transform  : tcgen05.ld D1 (the next chunk's load in flight) -> affine, PReLU, statistics, fp16 ->
//                 tcgen05.st back into the same tensor-memory buffer; one elected lane per warp arrives on the LEADER's barrier
//   warps 12-15   epilogue   : tcgen05.ld D2 -> fp16, staged 128 columns at a time (the resident weights leave room for half a row) in
//                 128-byte-swizzled boxes -> one TMA tensor store per box (UTMASTG), per-utterance column sums, row sums
// Tensor memory (per CTA, allocated with cta_group::2): D2 = columns 0-255; ring of 4 x 64 columns at 256-511 (D1, then q).
// Synchronisation: mbarriers only; barriers the leader's MMA thread waits on receive remote (cluster-scope) arrivals from
// the peer, MMA completion is multicast to both CTAs. Requires T >= 128 (a tile touches at most two utterances) and the
// plane layout of p (conv1's persistent kernels write it); otherwise the forward uses launch_tc_dconv's kernel.
#include <algorithm>
#include <cuda.h>
#include "kernels.h"
#include "tc_common.cuh"

namespace septfa {

namespace {

using namespace tc;


constexpr int kTileM = 128;
constexpr int kHalo = kPlaneHalo;                   // 4 = the largest dilation
constexpr int kSlabRows = kTileM + 2 * kHalo;       // 136 frames: tile + halo
constexpr int kPlaneBytes = kSlabRows * 16;         // 2176: one K-group (8 channels) of the slab
constexpr int kPChunkBytes = 4 * kPlaneBytes;       // 8704: 32 input channels
constexpr int kPStages = 4;
constexpr int kWHalfBytes = 128 * 128;              // 16 KB: this CTA's 128 output rows of one K-chunk (64) of the res_out image
constexpr int kTapHalfBytes = kDconvTapBytes / 2;   // 24 KB: [16 groups][3 taps][2 K halves][16 outputs x 8 inputs, fp16]
constexpr int kD1Bufs = 4;
constexpr int kOffW = 0;                                      // 1024-aligned (128B swizzle)
constexpr int kOffTap = kOffW + 8 * kWHalfBytes;
constexpr int kOffP = kOffTap + kTapHalfBytes;
constexpr int kOffSwc = kOffP + kPStages * kPChunkBytes;
constexpr int kOffEdge = kOffSwc + 4096;            // edge-correction tables: folded taps 0 and 2 [2][512] fp16 (exactly what the MMA multiplies by), beta1 / gamma1 [256] fp32
constexpr int kEdgeBytes = 2 * 512 * 2 + 256 * 4;
// (the edge corrections of a chunk, [8 rows][64 outputs] fp32, are written over the first 2 KB of the chunk's own p stage once the
// mini-GEMMs have read it: a table of their own per stage is what stood between three and four p stages)
constexpr int kEpiWarpBytes = 2 * 32 * 128;         // two staging boxes per epilogue warp: 32 rows x 64 fp16 columns, 128-byte-swizzled rows
constexpr int kOffEpi = (kOffEdge + kEdgeBytes + 1023) / 1024 * 1024;
constexpr int kOffBar = kOffEpi + 4 * kEpiWarpBytes;
constexpr int kSmemBytes = kOffBar + 512;
static_assert(kPStages <= 4, "barrier slots");
constexpr int kThreadsD = 16 * 32;
static_assert(kOffW % 1024 == 0 && kOffP % 16 == 0 && kSmemBytes <= 232448, "shared-memory plan");

struct DmParams {
  alignas(64) CUtensorMap racc_tmap;   // racc as a 2-D tensor [M rows][256 halves], box 64 columns x 32 rows, SWIZZLE_128B
  int M, T, ntiles, Mp, dil, discard;
  float slope2;
  double inv_n;                // 1 / (256 T), from the host (a double division on the device is a long software routine)
  const __half* p_planes;      // [32 K-groups][Mp slots][8 channels]; frame r lives in slot r + kHalo
  const Stat2* st_p;
  const uint8_t* tap_img2;     // [2 ranks][16 groups][3 taps][2 K halves][16 outputs x 8 inputs fp16]: per-CTA halves of the tap matrices
  const float4* swc;           // [256]: {sw[2i], sw[2i+1], c2f[2i], c2f[2i+1]}
  const float* w16;            // [3][512] the fp16-rounded folded taps as fp32 (edge corrections)
  const float* bog;            // [256] beta1 / gamma1
  const __half* w_img;         // res_out: 8 K-chunks x [256 rows x 128 B], 128B-swizzled
  __half* racc;                // [M,256]
  float* rowsum; double* colsum; Stat2* st_q;
};

// ---- cta_group::2 forms of the tcgen05 wrappers (tc_common.cuh has the cta_group::1 forms)
__device__ __forceinline__ void tmem_alloc2(uint32_t* slot, uint32_t ncols) {   // one warp of EACH CTA of the pair, same slot offset
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem, 256 rows over the pair] (+)= A[smem of each CTA: its 128 rows] * B[smem of each CTA: its half of N]^T
__device__ __forceinline__ void umma2_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(0u)
      : "memory");
}
// ... with the A operand in each CTA's tensor memory (its 128 rows = 128 lanes, 16-bit elements packed two per 32-bit
// column: element k of row m lives in lane m, column k / 2, low half for even k)
__device__ __forceinline__ void umma2_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(0u)
      : "memory");
}
// Arrive on the mbarrier at this offset in every CTA of `mask` when all previously issued MMAs of the pair have completed.
__device__ __forceinline__ void umma2_commit(uint64_t* bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
               "h"(mask)
               : "memory");
}
// Arrive on the barrier at this offset in CTA `rank` of the cluster (the caller's own CTA included). Default (CTA-scope)
// semantics, as in CUTLASS' ClusterBarrier::arrive(cta_id): what these barriers order are tensor-memory and async-proxy
// operations, which the tcgen05 fences around them govern; a cluster-scope release / acquire on every arrival and poll
// cost ~800 cycles per chunk in the MMA issuer.
__device__ __forceinline__ void mbar_arrive_cl(uint64_t* bar, uint32_t rank) {
  uint32_t remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(bar)), "r"(rank));
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
}
// The same without memory-ordering semantics: for arrivals that only hand tensor memory back (ordered by the tcgen05 fences).
// A release would first drain the thread's outstanding global stores.
__device__ __forceinline__ void mbar_arrive_cl_relaxed(uint64_t* bar, uint32_t rank) {
  uint32_t remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(bar)), "r"(rank));
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
}
// Non-blocking phase test (try_wait may suspend the thread for a system-dependent time when the phase is not complete).
__device__ __forceinline__ bool mbar_test_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// TMA tensor store of a 2-D box (SASS: UTMASTG), tracked by the thread's bulk async-group.
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* tmap, int c0, int c1, const void* ssrc) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];" ::"l"(tmap), "r"(c0), "r"(c1), "r"(smem_u32(ssrc))
               : "memory");
}
// One lane of a fully converged warp (elect.sync). The MMA issuers run their loops with the WHOLE warp (all lanes poll the
// barriers) and predicate the tcgen05 instructions on this: inside an `if (lane == 0)` region the compiler wraps every
// uniform-datapath instruction (UTCHMMA, UTCBAR) in its own elect / branch loop.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
// tcgen05.st without the wait (follow with tmem_st_wait())
__device__ __forceinline__ void tmem_st16_nowait(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
      "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptor, K-major, no swizzle: core matrices of 8 rows x 16 bytes (128 contiguous bytes);
// LBO = byte distance between core matrices adjacent in K, SBO = between core matrices adjacent in M / N.
__device__ __forceinline__ uint64_t make_ns_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;
  return d;
}

template <bool AMAX>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreadsD, 1) k_dconv_mma2(const __grid_constant__ DmParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kOffBar);
  uint64_t* w_full = bars;            // [8] bulk-copy bytes: this CTA's half of weight chunk j (once)
  uint64_t* w_peer = bars + 8;        // [8] leader: the peer's half of chunk j has landed (relay)
  uint64_t* tap_full = bars + 16;     //     bulk-copy bytes (once)
  uint64_t* tap_peer = bars + 17;     //     leader: relay
  uint64_t* p_full = bars + 18;       // [kPStages <= 4] bulk-copy bytes
  uint64_t* p_peer = bars + 22;       // [kPStages] leader: the peer's slab has landed (relay)
  uint64_t* p_empty = bars + 26;      // [kPStages] mini-MMA commit (multicast) + one lane of the 4 local transform warps of the chunk + the edge warp
  uint64_t* corr_full = bars + 30;    // [kPStages] the edge warp has written the corrections of the chunk in this p stage
  uint64_t* d1_full = bars + 34;      // [4] mini-MMA commit (multicast)
  uint64_t* d1_empty = bars + 38;     // [4] leader: res_out MMA commit (the buffer held D1, then q)
  uint64_t* a2_full = bars + 42;      // [4] leader: the 8 transform warps of the pair that take this chunk (q is in tensor memory)
  uint64_t* d2_full = bars + 46;      //     MMA commit (multicast)
  uint64_t* d2_empty = bars + 47;     //     leader: 8 epilogue warps of the pair
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 48);
  uint64_t* ms_full = bars + 49;      // [2] the edge warp has published mean / rstd of the tile's utterances (by tile parity)
  float4* ms_s = reinterpret_cast<float4*>(bars + 52);   // [2] {mean0, rstd0, mean1, rstd1}
  constexpr uint32_t IDESC_MAIN = make_idesc_f16(2 * kTileM, 256);
  constexpr uint32_t IDESC_MINI = make_idesc_f16(2 * kTileM, 32);

  // Role index, not the hardware warp id: the SM's warp arbiter prefers the highest warp ids, so the single-thread roles
  // (loaders, MMA issuers, relay / edge warp) sit on hardware warps 12-15, the transform on 0-7, the epilogue on 8-11.
  // The shift by 4 keeps role % 4 == hardware warp % 4 (the tensor-memory lane quarter a warp may access).
  const int warp = ((threadIdx.x >> 5) + 4) & 15, lane = threadIdx.x & 31;
  const uint32_t crank = cluster_ctarank();
  const bool leader = crank == 0;
  if (threadIdx.x == 0) {
    if ((smem_u32(smem) & 1023u) != 0u) __trap();
    for (int j = 0; j < 8; ++j) { mbar_init(w_full + j, 1); mbar_init(w_peer + j, 1); }
    mbar_init(tap_full, 1); mbar_init(tap_peer, 1);
    for (int s = 0; s < kPStages; ++s) { mbar_init(p_full + s, 1); mbar_init(p_peer + s, 1); mbar_init(p_empty + s, 6); mbar_init(corr_full + s, 1); }
    for (int s = 0; s < kD1Bufs; ++s) { mbar_init(d1_full + s, 1); mbar_init(d1_empty + s, 1); mbar_init(a2_full + s, 8); }
    mbar_init(d2_full, 1); mbar_init(d2_empty, 8);
    mbar_init(ms_full, 1); mbar_init(ms_full + 1, 1);
    fence_mbar_init();
  }
  if (warp == 2) tmem_alloc2(tmem_slot, 512);
  {
    __half* edge_w = reinterpret_cast<__half*>(smem + kOffEdge);
    edge_w[threadIdx.x] = __float2half_rn(__ldg(p.w16 + threadIdx.x));                    // tap 0 (fp16 values stored as fp32: exact)
    edge_w[kH + threadIdx.x] = __float2half_rn(__ldg(p.w16 + 2 * kH + threadIdx.x));      // tap 2
    if (threadIdx.x < kC) reinterpret_cast<float*>(smem + kOffEdge + 4 * kH)[threadIdx.x] = __ldg(p.bog + threadIdx.x);
  }
  __syncthreads();
  if (warp == 1 && lane == 0) {
    // static weights, once, before the dependency wait: this CTA's half of every tap matrix and of the res_out image
    mbar_expect_tx(tap_full, kTapHalfBytes);
    bulk_copy_g2s(smem + kOffTap, p.tap_img2 + (size_t)crank * kTapHalfBytes, kTapHalfBytes, tap_full);
    for (int j = 0; j < 8; ++j) {   // rows 128 r .. 128 r + 127 of chunk j: 16 KB contiguous
      mbar_expect_tx(w_full + j, kWHalfBytes);
      bulk_copy_g2s(smem + kOffW + j * kWHalfBytes, reinterpret_cast<const uint8_t*>(p.w_img) + (size_t)j * 2 * kWHalfBytes + (size_t)crank * kWHalfBytes,
                    kWHalfBytes, w_full + j);
    }
  }
  pdl_wait();   // everything below reads what earlier kernels of the chain wrote
  tc_fence_before();
  cluster_sync_all();   // (also a CTA barrier) both CTAs' mbarriers are initialised and their tensor memory is allocated
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // the pair walks tile pairs: cluster c takes pairs c, c + nclusters, ...; rank r the tile 2 * pair + r. Both CTAs run
  // the same number of tiles (the last pair of an odd tile count has an empty tile: no valid rows, nothing stored).
  const int npairs = (p.ntiles + 1) / 2;
  const int first_pair = (int)blockIdx.x / 2, pair_stride = (int)gridDim.x / 2;
  const int my_tiles = first_pair < npairs ? (npairs - first_pair + pair_stride - 1) / pair_stride : 0;
  const int first = 2 * first_pair + (int)crank, stride = 2 * pair_stride, tile_end = 2 * npairs;

  if (warp == 0) {
    // ------------------------------------------------------------ p loader (K-group planes, tile + halo)
    {
      auto discard_chunk = [&](int gp) {   // whole warp: the 60 lines (4 planes x 15) of chunk gp that no other tile reads
        const int tp = first + (gp >> 3) * stride, jp = gp & 7;
        if (p.discard && (tp + 1) * kTileM <= p.M) {
#pragma unroll
          for (int q = 0; q < 2; ++q) {
            const int idx = lane + 32 * q;
            if (idx < 60) {
              const int kg = idx / 15, ln = 1 + idx % 15;
              const __half* a = p.p_planes + ((size_t)(jp * 4 + kg) * p.Mp + (size_t)tp * kTileM) * 8 + ln * 64;
              asm volatile("discard.global.L2 [%0], 128;" ::"l"(a) : "memory");
            }
          }
        }
      };
      int g = 0;
      for (int tile = first; tile < tile_end; tile += stride) {
        for (int j = 0; j < 8; ++j, ++g) {
          const int s = g % kPStages, u = g / kPStages;
          if (u > 0) {
            mbar_wait(p_empty + s, (u - 1) & 1, 100 + j);
            // The chunk that held this stage (kPStages back) is consumed, and p is read exactly once: its lines are dead but dirty
            // (conv1 wrote them) - they would sit in the L2 until evicted and then be written to DRAM. discard.L2 drops them, which
            // leaves the L2 to the residual stream. Only the 15 lines per plane no other tile reads (frames r0 + 4 .. r0 + 123:
            // the neighbours' halos are the first and the last line), and never a tile with rows past M (their slots are the
            // zero padding that no kernel rewrites).
            discard_chunk(g - kPStages);
          }
          if (lane == 0) {
            mbar_expect_tx(p_full + s, kPChunkBytes);
#pragma unroll
            for (int kg = 0; kg < 4; ++kg)   // frames r0 - 4 .. r0 + 131 = slots r0 .. r0 + 135
              bulk_copy_g2s(smem + kOffP + s * kPChunkBytes + kg * kPlaneBytes,
                            p.p_planes + ((size_t)(j * 4 + kg) * p.Mp + (size_t)tile * kTileM) * 8, kPlaneBytes, p_full + s);
          }
          __syncwarp();
        }
      }
      for (int gp = max(0, g - kPStages); gp < g; ++gp) {   // the chunks still in the ring when the loop ends
        mbar_wait(p_empty + gp % kPStages, (gp / kPStages) & 1, 110);
        discard_chunk(gp);
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ------------------------------------------------------------ edge warp: zero padding of the NORMALISED signal.
    // The tensor-core convolution reads whatever neighbours the shifted view holds; for the <= 2 * dil rows of a tile whose
    // tap falls outside their utterance this warp computes what that tap contributed,
    //   corr[o] = w'_k[o] * ((p_wrong[c] - mean) + (beta / gamma)[c] / rstd)        (c = o / 2, the same fp16 operands the MMA saw),
    // into a small table per p stage; the transform lane that owns such a row subtracts its 32 entries. (Done inside the
    // transform warps - 170 divergent instructions per chunk and side - these few rows set the pace of the whole pair.)
    // lane -> (slot = lane / 4, K-group = lane % 4); slots 0-3: rows T - 4 .. T - 1 of an utterance (tap +dil invalid),
    // slots 4-7: rows 0 .. 3 (tap -dil invalid). With T >= 128 a tile holds at most one group of each kind.
    const __half* edge_w = reinterpret_cast<const __half*>(smem + kOffEdge);
    const float* edge_bog = reinterpret_cast<const float*>(smem + kOffEdge + 4 * kH);
    const double inv_n = p.inv_n;
    const int slot = lane >> 2, part = lane & 3;
    int g = 0, lt = 0;
    for (int tile = first; tile < tile_end; tile += stride, ++lt) {
      const int r0 = tile * kTileM, nrows = max(0, min(kTileM, p.M - r0));
      const int b_first = r0 / p.T, e1 = (b_first + 1) * p.T;
      float2 mr = make_float2(0.f, 1.f);
      if (nrows > 0 && lane < 2 && (lane == 0 || e1 < r0 + nrows)) mr = stat_mean_rstd(p.st_p + b_first + lane, inv_n, 1e-8f);
      const float m0 = __shfl_sync(0xffffffffu, mr.x, 0), s0 = __shfl_sync(0xffffffffu, mr.y, 0);
      const float m1 = __shfl_sync(0xffffffffu, mr.x, 1), s1 = __shfl_sync(0xffffffffu, mr.y, 1);
      // ... published for the transform warps: this warp runs up to a p ring ahead of them, they are the pair's critical path at
      // a tile boundary and the statistics cost two L2 round trips plus double arithmetic. (Slot lt & 1 was last read at the top
      // of tile lt - 2; this warp gets here only after the transform has released chunk 4 of tile lt - 1.)
      if (lane == 0) { ms_s[lt & 1] = make_float4(m0, s0, m1, s1); mbar_arrive(ms_full + (lt & 1)); }
      // the row of this lane's slot (if the tile has it) and its utterance
      int row = -1; bool second = false;
      if (slot < 4) {                       // t = T - i, i = 4 - slot: invalid iff i <= dil
        const int i = 4 - slot;
        if (i <= p.dil) {
          if (e1 - i >= r0 && e1 - i < r0 + nrows) row = e1 - i;
          else if (e1 + p.T - i >= r0 && e1 + p.T - i < r0 + nrows) { row = e1 + p.T - i; second = true; }
        }
      } else {                              // t = slot - 4: invalid iff t < dil
        const int t = slot - 4;
        if (t < p.dil) {
          if (b_first * p.T + t >= r0 && b_first * p.T + t < r0 + nrows) row = b_first * p.T + t;
          else if (e1 + t >= r0 && e1 + t < r0 + nrows) { row = e1 + t; second = true; }
        }
      }
      const float mean = second ? m1 : m0, inv_rstd = 1.0f / (second ? s1 : s0);
      const int srow = kHalo + (row - r0) + (slot < 4 ? p.dil : -p.dil);
      const __half* wk_side = edge_w + (slot < 4 ? kH : 0);   // tap 2 for the rows at an utterance's end, tap 0 at its start
      const bool any_row = __any_sync(0xffffffffu, row >= 0);
      for (int j = 0; j < 8; ++j, ++g) {
        const int sp = g % kPStages;
        mbar_wait(p_full + sp, (g / kPStages) & 1, 140 + j);
        if (any_row) {
          float cv[16];
          if (row >= 0) {
            const uint4 raw = *reinterpret_cast<const uint4*>(smem + kOffP + sp * kPChunkBytes + part * kPlaneBytes + srow * 16);
            const uint32_t rw[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
            for (int e2 = 0; e2 < 4; ++e2) {
              const float2 pv = __half22float2(*reinterpret_cast<const __half2*>(&rw[e2]));
              const int c = part * 8 + e2 * 2;     // input channel within the chunk's 32
              const float2 bg = *reinterpret_cast<const float2*>(edge_bog + j * 32 + c);
              const float u0 = (pv.x - mean) + bg.x * inv_rstd, u1 = (pv.y - mean) + bg.y * inv_rstd;
              const uint2 wr = *reinterpret_cast<const uint2*>(wk_side + j * 64 + 2 * c);
              const float2 w01 = __half22float2(*reinterpret_cast<const __half2*>(&wr.x)), w23 = __half22float2(*reinterpret_cast<const __half2*>(&wr.y));
              cv[4 * e2] = w01.x * u0; cv[4 * e2 + 1] = w01.y * u0; cv[4 * e2 + 2] = w23.x * u1; cv[4 * e2 + 3] = w23.y * u1;
            }
          }
          // the table goes over the start of the stage itself, as soon as the mini-GEMMs of the chunk (both CTAs: multicast commit)
          // have read it; the transform warps wait for their own tensor-memory loads meanwhile
          mbar_wait(d1_full + (g % kD1Bufs), (g / kD1Bufs) & 1, 150 + j);
          if (row >= 0) {
            float4* dst = reinterpret_cast<float4*>(smem + kOffP + sp * kPChunkBytes + slot * 256 + part * 64);
#pragma unroll
            for (int e = 0; e < 4; ++e) dst[e] = make_float4(cv[4 * e], cv[4 * e + 1], cv[4 * e + 2], cv[4 * e + 3]);
          }
          fence_proxy_async();   // generic-proxy writes into a stage the next bulk copy will overwrite
        }
        __syncwarp();
        if (lane == 0) { mbar_arrive(corr_full + sp); mbar_arrive(p_empty + sp); }
      }
    }
  } else if (warp == 3) {
    if (!leader) {
      // ---------------------------------------------------------- relay (peer CTA): tell the leader what has landed here
      if (lane == 0) {
        mbar_wait(tap_full, 0, 160);
        mbar_arrive_cl(tap_peer, 0);
        const int total = my_tiles * 8;
        for (int g = 0; g < max(total, 8); ++g) {
          if (g < 8) { mbar_wait(w_full + g, 0, 170 + g); mbar_arrive_cl(w_peer + g, 0); }
          if (g < total) {
            const int s = g % kPStages, u = g / kPStages;
            mbar_wait(p_full + s, u & 1, 180);
            mbar_arrive_cl(p_peer + s, 0);
          }
        }
      }
    } else {
      // ---------------------------------------------------------- depthwise mini-GEMM issuer (leader CTA). A thread of its own:
      // issuing a tcgen05.mma costs its thread ~100 cycles whatever the shape, so one thread issuing the 6 mini-MMAs and the 4
      // res_out MMAs of a chunk (~1.7 k cycles) set the pace of the whole pair.
      mbar_wait(tap_full, 0, 190);
      mbar_wait(tap_peer, 0, 191);
      const int total = my_tiles * 8;
      for (int gi = 0; gi < total; ++gi) {
        // chunk gi -> D1[gi % 4] of both CTAs
        const int sp = gi % kPStages, up = gi / kPStages, b = gi % kD1Bufs, ub = gi / kD1Bufs, j = gi & 7;
        mbar_wait(p_full + sp, up & 1, 200 + j);
        mbar_wait(p_peer + sp, up & 1, 205 + j);
        if (ub > 0) mbar_wait(d1_empty + b, (ub - 1) & 1, 210 + j);
        tc_fence_after();
        const uint32_t slab = smem_u32(smem + kOffP + sp * kPChunkBytes);
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < 3; ++k) {       // tap-major: consecutive MMAs accumulate into different columns
#pragma unroll
            for (int grp = 0; grp < 2; ++grp) {
              const uint32_t a_addr = slab + (uint32_t)(grp * 2 * kPlaneBytes + (kHalo + (k - 1) * p.dil) * 16);
              const uint32_t b_addr = smem_u32(smem + kOffTap + ((j * 2 + grp) * 3 + k) * 512);
              umma2_f16(tmem_base + 256u + (uint32_t)(b * 64 + grp * 32), make_ns_desc(a_addr, (uint32_t)kPlaneBytes, 128u),
                        make_ns_desc(b_addr, 256u, 128u), IDESC_MINI, k != 0);
            }
          }
          umma2_commit(d1_full + b, (uint16_t)3);
          umma2_commit(p_empty + sp, (uint16_t)3);
        }
        __syncwarp();
      }
    }
    __syncwarp();
  } else if (warp == 2) {
    // ------------------------------------------------------------ res_out MMA issuer (leader CTA)
    if (leader) {
      const int total = my_tiles * 8;
      for (int gm = 0; gm < total; ++gm) {
        const int j = gm & 7, lt = gm >> 3, ba = gm % kD1Bufs, ua = gm / kD1Bufs;
        if (j == 0 && lt > 0) mbar_wait(d2_empty, (lt - 1) & 1, 220);
        if (lt == 0) { mbar_wait(w_full + j, 0, 230 + j); mbar_wait(w_peer + j, 0, 235 + j); }
        mbar_wait(a2_full + ba, ua & 1, 240 + j);
        tc_fence_after();
        const uint32_t a_tmem = tmem_base + 256u + (uint32_t)(ba * 64);   // q: K 0..31 at +0..15, K 32..63 at +32..47
        const uint64_t b_desc = make_sw128_desc(smem_u32(smem + kOffW + j * kWHalfBytes));
        if (elect_one()) {
#pragma unroll
        for (int kk = 0; kk < 4; ++kk)
          umma2_f16_ts(tmem_base, a_tmem + (uint32_t)((kk >> 1) * 32 + (kk & 1) * 8), b_desc + (uint64_t)(kk * 2), IDESC_MAIN, (j | kk) != 0);
        umma2_commit(d1_empty + ba, (uint16_t)1);
        if (j == 7) umma2_commit(d2_full, (uint16_t)3);
        }
        __syncwarp();
      }
    }
    __syncwarp();
  } else if (warp >= 4 && warp < 12) {
    // ------------------------------------------------------------ transform: D1 -> q -> A2
    const int q4 = warp & 3, par = (warp - 4) >> 2;      // TMEM lane quarter (hardware: warp % 4), parity of the chunks this warp takes
    const int rl = q4 * 32 + lane;                        // a lane = a row of the tile
    const float2 sl2 = make_float2(p.slope2, p.slope2);
    float2* k0_s = reinterpret_cast<float2*>(smem + kOffSwc);   // [2 utterances of the tile][256 output pairs]
    const int tt = (warp - 4) * 32 + lane;                      // this thread's output pair when the table is built
    const float4 t4 = __ldg(p.swc + tt);                         // tile-invariant: sums of the fp16 taps, folded constants
    int g = 0, lt = 0;
    for (int tile = first; tile < tile_end; tile += stride, ++lt) {
      const int r0 = tile * kTileM, nrows = max(0, min(kTileM, p.M - r0));
      const int b_first = r0 / p.T, e1 = (b_first + 1) * p.T;   // first row of the tile's second utterance
      // mean / rstd of the tile's (at most two) utterances come from the edge warp, which runs ahead: at a tile boundary these
      // warps are the pair's critical path (the first res_out MMA of a tile waits for their first chunk)
      mbar_wait(ms_full + (lt & 1), (lt >> 1) & 1, 320);
      const float4 ms4 = ms_s[lt & 1];
      const float m0 = ms4.x, s0 = ms4.y, m1 = ms4.z, s1 = ms4.w;
      const int row = r0 + rl;
      const bool valid = rl < nrows, second = row >= e1;
      const float mean = second ? m1 : m0, rstd = second ? s1 : s0;
      const int t = row - (second ? e1 : b_first * p.T);
      // rows whose tap falls outside their utterance: slot of the edge warp's correction table (-1: none)
      const int cslot = !valid ? -1 : (t < p.dil ? 4 + t : (p.T - t <= p.dil ? 4 - (p.T - t) : -1));
      const float2 rs2 = make_float2(rstd, rstd);
      // the additive part of the affine, c2f - rstd * mean * sw, depends on the row only through its utterance: one table
      // per tile (two utterances x 512 outputs) instead of one FFMA2 per pair and row (the transform is bound by the FP32 pipe)
      asm volatile("bar.sync 1, 256;" ::: "memory");            // every transform warp is done with the previous tile's table
      {
        k0_s[tt] = __ffma2_rn(make_float2(-m0 * s0, -m0 * s0), make_float2(t4.x, t4.y), make_float2(t4.z, t4.w));
        k0_s[256 + tt] = __ffma2_rn(make_float2(-m1 * s1, -m1 * s1), make_float2(t4.x, t4.y), make_float2(t4.z, t4.w));
      }
      asm volatile("bar.sync 1, 256;" ::: "memory");
      const float2* k0_row = k0_s + (second ? 256 : 0);
      float2 accS = make_float2(0.f, 0.f), accQ = make_float2(0.f, 0.f);
      auto t_addr = [&](int gg, int hf) { return tmem_base + 256u + (uint32_t)((gg % kD1Bufs) * 64 + hf * 32) + ((uint32_t)(q4 * 32) << 16); };
      // half a chunk: v (the fp32 depthwise accumulators of this lane's row, 32 outputs) -> q (fp16 pairs) -> tensor memory
      auto half_chunk = [&](uint32_t (&u)[32], int j, int gg, int hf) {
        const float2* kk0 = k0_row + j * 32 + hf * 16;
        uint32_t h[16];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const float2 x = __ffma2_rn(rs2, make_float2(__uint_as_float(u[8 * i + 2 * k]), __uint_as_float(u[8 * i + 2 * k + 1])),
                                        kk0[i * 4 + k]);   // (same address in every lane of one utterance: broadcast)
            const float2 ax = __fmul2_rn(sl2, x);
            float2 qv;
            if constexpr (AMAX) qv = make_float2(fmaxf(x.x, ax.x), fmaxf(x.y, ax.y));
            else qv = make_float2(fminf(x.x, ax.x), fminf(x.y, ax.y));
            accS = __fadd2_rn(accS, qv);
            accQ = __ffma2_rn(qv, qv, accQ);
            h[i * 4 + k] = pack_half2(qv.x, qv.y);
          }
        }
        tmem_st16_nowait(t_addr(gg, hf), h);   // q (fp16 pairs) over the first 16 of the 32 columns that were read
      };
      // The two warps of a lane quarter take ALTERNATE chunks (all 64 columns each) instead of half of every chunk: the
      // transform is bound by the FP32 pipe of its SM sub-partition, and two warps in lock step (same barrier, same
      // instruction mix) fight for it during the arithmetic and leave it idle during their tensor-memory round trips.
      uint32_t va[32], vb[32];
#pragma unroll 1
      for (int j = par; j < 8; j += 2) {
        const int gg = g + j, sp = gg % kPStages;
        mbar_wait(d1_full + (gg % kD1Bufs), (gg / kD1Bufs) & 1, 300 + j);
        tc_fence_after();
        tmem_ld32_nowait(t_addr(gg, 0), va);
        tmem_ld32_nowait(t_addr(gg, 1), vb);
        tmem_ld_wait();
        if (cslot >= 0) {
          // zero padding of the normalised signal: take back what the out-of-utterance tap contributed (edge warp's table)
          mbar_wait(corr_full + sp, (gg / kPStages) & 1, 310 + j);
          const float4* cr = reinterpret_cast<const float4*>(smem + kOffP + sp * kPChunkBytes + cslot * 256);   // over the consumed stage
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const float4 c4 = cr[e], d4 = cr[8 + e];
            va[4 * e] = __float_as_uint(__uint_as_float(va[4 * e]) - c4.x);
            va[4 * e + 1] = __float_as_uint(__uint_as_float(va[4 * e + 1]) - c4.y);
            va[4 * e + 2] = __float_as_uint(__uint_as_float(va[4 * e + 2]) - c4.z);
            va[4 * e + 3] = __float_as_uint(__uint_as_float(va[4 * e + 3]) - c4.w);
            vb[4 * e] = __float_as_uint(__uint_as_float(vb[4 * e]) - d4.x);
            vb[4 * e + 1] = __float_as_uint(__uint_as_float(vb[4 * e + 1]) - d4.y);
            vb[4 * e + 2] = __float_as_uint(__uint_as_float(vb[4 * e + 2]) - d4.z);
            vb[4 * e + 3] = __float_as_uint(__uint_as_float(vb[4 * e + 3]) - d4.w);
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(p_empty + sp);
        half_chunk(va, j, gg, 0);
        half_chunk(vb, j, gg, 1);
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cl(a2_full + (gg % kD1Bufs), 0);   // one arrival per warp, on the leader's barrier
      }
      g += 8;
      // statistics of q of this warp's 32 rows x 256 columns, per utterance: fixed-order shuffle trees, double atomics
      const float sv = valid ? accS.x + accS.y : 0.f, qv = valid ? accQ.x + accQ.y : 0.f;
      // (an utterance boundary falls into one warp's 32 rows of few tiles: two shuffle trees instead of four elsewhere)
      const unsigned secm = __ballot_sync(0xffffffffu, second);
      float a0 = 0.f, c0 = 0.f, a1 = 0.f, c1 = 0.f;
      if (secm == 0u) { a0 = warp_sum(sv); c0 = warp_sum(qv); }
      else if (secm == 0xffffffffu) { a1 = warp_sum(sv); c1 = warp_sum(qv); }
      else {
        a0 = warp_sum(second ? 0.f : sv); c0 = warp_sum(second ? 0.f : qv);
        a1 = warp_sum(second ? sv : 0.f); c1 = warp_sum(second ? qv : 0.f);
      }
      if (lane == 0 && nrows > 0) {
        if (secm != 0xffffffffu) {
          atomicAdd(&p.st_q[b_first].s, (double)a0);
          atomicAdd(&p.st_q[b_first].ss, (double)c0);
        }
        if (secm != 0u && e1 < r0 + nrows) {
          atomicAdd(&p.st_q[b_first + 1].s, (double)a1);
          atomicAdd(&p.st_q[b_first + 1].ss, (double)c1);
        }
      }
    }
  } else if (warp >= 12) {
    // ------------------------------------------------------------ epilogue: D2 -> racc (fp16), row / column sums
    // The resident weights leave room to stage HALF a row per lane: the accumulator's two 128-column halves go through the
    // same buffer, two boxes of 32 rows x 64 columns per warp in the TMA 128-byte-swizzle layout (a lane = a row writes its
    // 16-byte pieces conflict-free), and leave with ONE tensor-map store per box: 16 TMA requests per CTA and tile. (One
    // 256-byte bulk store per row and half = 256 requests per tile kept the SM's TMA unit busy for ~5 k cycles per half.)
    const int q4 = warp & 3;
    const int rl = q4 * 32 + lane;
    uint8_t* box_w = smem + kOffEpi + (warp - 12) * kEpiWarpBytes;   // [2 boxes][32 rows][128 B], 1024-aligned
    const uint32_t rsw = (uint32_t)(lane & 7);
    int lt = 0;
    for (int tile = first; tile < tile_end; tile += stride, ++lt) {
      const int r0 = tile * kTileM, nrows = max(0, min(kTileM, p.M - r0));
      const int b_first = r0 / p.T, e1 = (b_first + 1) * p.T;
      const int row = r0 + rl;
      const bool valid = rl < nrows;
      const int nv_w = max(0, min(32, nrows - q4 * 32));               // valid rows of this warp
      const int n0_w = max(0, min(nv_w, e1 - (r0 + q4 * 32)));         // ... that belong to the tile's first utterance
      mbar_wait(d2_full, lt & 1, 500);
      tc_fence_after();
      float2 racc2 = make_float2(0.f, 0.f);
      const uint32_t t_row = tmem_base + ((uint32_t)(q4 * 32) << 16);
      auto pack_store = [&](const uint32_t (&u)[32], int cc) {   // cc: 32-column piece within the staged half row
        uint8_t* dst = box_w + (cc >> 1) * 4096 + lane * 128;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float v8[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) v8[e] = __uint_as_float(u[8 * i + e]);
          racc2 = __fadd2_rn(racc2, __fadd2_rn(__fadd2_rn(make_float2(v8[0], v8[1]), make_float2(v8[2], v8[3])),
                                               __fadd2_rn(make_float2(v8[4], v8[5]), make_float2(v8[6], v8[7]))));
          *reinterpret_cast<uint4*>(dst + ((((uint32_t)((cc & 1) * 4 + i)) ^ rsw) << 4)) =
              make_uint4(pack_half2(v8[0], v8[1]), pack_half2(v8[2], v8[3]), pack_half2(v8[4], v8[5]), pack_half2(v8[6], v8[7]));
        }
      };
      // the staged half (two boxes) leaves with one tensor store per box
      auto store_half = [&](int hh) {
        fence_proxy_async();             // our generic-proxy stores -> visible to the tensor store
        __syncwarp();
        if (lane == 0 && nv_w > 0) {       // rows past M are clipped by the tensor map
          tma_store_2d(&p.racc_tmap, hh * 128, r0 + q4 * 32, box_w);
          tma_store_2d(&p.racc_tmap, hh * 128 + 64, r0 + q4 * 32, box_w + 4096);
          bulk_commit_group();
        }
      };
      // per-utterance column sums of this warp's rows (from the staged fp16 values): lane -> 4 columns of one box
      auto colsum_half = [&](int hh) {
        float2 c0[2], c1[2];
#pragma unroll
        for (int e = 0; e < 2; ++e) c0[e] = c1[e] = make_float2(0.f, 0.f);
        const uint8_t* colb = box_w + (lane >> 4) * 4096 + (lane & 1) * 8;
        const uint32_t c16 = (uint32_t)((lane & 15) >> 1);
        if (nv_w == 32 && (n0_w == 32 || n0_w == 0)) {
          // all 32 rows belong to one utterance (every warp but the one on an utterance boundary / the tensor's end): rows
          // are first added four at a time as fp16 pairs, then accumulated in fp32 - a third of the instructions of the
          // general path below, in independent chains. (The fp16 partial sums round like racc itself does, and the column
          // MEANS over >= 128 frames average those roundings away.)
          float2 f0 = make_float2(0.f, 0.f), f1 = f0, g0 = f0, g1 = f0;
#pragma unroll
          for (int r4 = 0; r4 < 32; r4 += 4) {
            uint2 raw[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) raw[k] = *reinterpret_cast<const uint2*>(colb + (r4 + k) * 128 + ((c16 ^ (uint32_t)((r4 + k) & 7)) << 4));
            const __half2 lo = __hadd2(__hadd2(*reinterpret_cast<const __half2*>(&raw[0].x), *reinterpret_cast<const __half2*>(&raw[1].x)),
                                       __hadd2(*reinterpret_cast<const __half2*>(&raw[2].x), *reinterpret_cast<const __half2*>(&raw[3].x)));
            const __half2 hi = __hadd2(__hadd2(*reinterpret_cast<const __half2*>(&raw[0].y), *reinterpret_cast<const __half2*>(&raw[1].y)),
                                       __hadd2(*reinterpret_cast<const __half2*>(&raw[2].y), *reinterpret_cast<const __half2*>(&raw[3].y)));
            if (r4 & 4) { g0 = __fadd2_rn(g0, __half22float2(lo)); g1 = __fadd2_rn(g1, __half22float2(hi)); }
            else { f0 = __fadd2_rn(f0, __half22float2(lo)); f1 = __fadd2_rn(f1, __half22float2(hi)); }
          }
          f0 = __fadd2_rn(f0, g0);
          f1 = __fadd2_rn(f1, g1);
          if (n0_w == 32) { c0[0] = f0; c0[1] = f1; } else { c1[0] = f0; c1[1] = f1; }
        } else {
#pragma unroll 1
          for (int r4 = 0; r4 < nv_w; r4 += 4) {
            uint2 raw[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const int r = min(r4 + k, 31);
              raw[k] = *reinterpret_cast<const uint2*>(colb + r * 128 + ((c16 ^ (uint32_t)(r & 7)) << 4));
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const int r = r4 + k;
              const float2 lo = __half22float2(*reinterpret_cast<const __half2*>(&raw[k].x)), hi = __half22float2(*reinterpret_cast<const __half2*>(&raw[k].y));
              if (r < n0_w) { c0[0] = __fadd2_rn(c0[0], lo); c0[1] = __fadd2_rn(c0[1], hi); }
              else if (r < nv_w) { c1[0] = __fadd2_rn(c1[0], lo); c1[1] = __fadd2_rn(c1[1], hi); }
            }
          }
        }
        double* cdst = p.colsum + (size_t)b_first * kC + hh * 128 + lane * 4;
        if (n0_w > 0) {
#pragma unroll
          for (int e = 0; e < 2; ++e) { atomicAdd(cdst + 2 * e, (double)c0[e].x); atomicAdd(cdst + 2 * e + 1, (double)c0[e].y); }
        }
        if (nv_w > n0_w) {
          cdst += kC;
#pragma unroll
          for (int e = 0; e < 2; ++e) { atomicAdd(cdst + 2 * e, (double)c1[e].x); atomicAdd(cdst + 2 * e + 1, (double)c1[e].y); }
        }
        __syncwarp();                    // every lane's column-sum reads of the staging boxes are done
      };
      // The whole accumulator leaves tensor memory in ONE software pipeline (a 32-column load in flight behind every
      // conversion), because nothing else of this role is on the pair's critical path: the first res_out MMA of the next tile
      // waits for D2. Columns 0-127 go to the staging boxes as fp16, columns 128-255 wait in REGISTERS as fp16 pairs, so that
      // D2 goes back to the MMA warp before the tensor stores, the column sums of either half and the staging of the second
      // (waiting for those held the accumulator for 3.5-6 k cycles per tile; the unpipelined second half for 2.1 k).
      uint32_t h2[64];
      auto keep = [&](const uint32_t (&u)[32], int c) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float v8[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) v8[e] = __uint_as_float(u[8 * i + e]);
          racc2 = __fadd2_rn(racc2, __fadd2_rn(__fadd2_rn(make_float2(v8[0], v8[1]), make_float2(v8[2], v8[3])),
                                               __fadd2_rn(make_float2(v8[4], v8[5]), make_float2(v8[6], v8[7]))));
#pragma unroll
          for (int e = 0; e < 4; ++e) h2[c * 16 + i * 4 + e] = pack_half2(v8[2 * e], v8[2 * e + 1]);
        }
      };
      {
        uint32_t va[32], vb[32];
        tmem_ld32_nowait(t_row, va);
        if (lane == 0) bulk_wait_read_all();   // the previous tile's boxes have left the staging buffer
        __syncwarp();
        tmem_ld_wait();
        tmem_ld32_nowait(t_row + 32u, vb);
        pack_store(va, 0);
        tmem_ld_wait();
        tmem_ld32_nowait(t_row + 64u, va);
        pack_store(vb, 1);
        tmem_ld_wait();
        tmem_ld32_nowait(t_row + 96u, vb);
        pack_store(va, 2);
        tmem_ld_wait();
        tmem_ld32_nowait(t_row + 128u, va);
        pack_store(vb, 3);
        tmem_ld_wait();
        tmem_ld32_nowait(t_row + 160u, vb);
        keep(va, 0);
        tmem_ld_wait();
        tmem_ld32_nowait(t_row + 192u, va);
        keep(vb, 1);
        tmem_ld_wait();
        tmem_ld32_nowait(t_row + 224u, vb);
        keep(va, 2);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cl(d2_empty, 0);   // every column is in registers or staged
        keep(vb, 3);
      }
      store_half(0);   // the staged half (two boxes) leaves with one tensor store per box
      colsum_half(0);
      if (lane == 0) bulk_wait_read_all();   // the first half's boxes have left the staging buffer
      __syncwarp();
#pragma unroll
      for (int cc = 0; cc < 4; ++cc) {
        uint8_t* dst = box_w + (cc >> 1) * 4096 + lane * 128;
#pragma unroll
        for (int i = 0; i < 4; ++i)
          *reinterpret_cast<uint4*>(dst + ((((uint32_t)((cc & 1) * 4 + i)) ^ rsw) << 4)) =
              make_uint4(h2[cc * 16 + i * 4], h2[cc * 16 + i * 4 + 1], h2[cc * 16 + i * 4 + 2], h2[cc * 16 + i * 4 + 3]);
      }
      store_half(1);
      colsum_half(1);
      if (valid) p.rowsum[row] = racc2.x + racc2.y;
    }
    if (lane == 0) bulk_wait_read_all();
    __syncwarp();
  }

  tc_fence_before();
  cluster_sync_all();   // neither CTA leaves (or frees its tensor memory) while the pair's MMAs may still touch it
  if (warp == 2) tmem_dealloc2(tmem_base, 512);
}

}  // namespace

cudaError_t dconv_mma2_setup() {
  cudaError_t e = cudaFuncSetAttribute(k_dconv_mma2<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
  if (e != cudaSuccess) return e;
  return cudaFuncSetAttribute(k_dconv_mma2<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
}

void launch_dconv_mma2(const DconvMmaParams& c, cudaStream_t st) {
  DmParams p{};
  p.M = c.M; p.T = c.T; p.ntiles = (c.M + kTileM - 1) / kTileM; p.Mp = c.Mp; p.dil = c.dil; p.slope2 = c.slope2; p.discard = c.discard; p.inv_n = 1.0 / ((double)kC * c.T);
  p.p_planes = c.p_planes; p.st_p = c.st_p; p.tap_img2 = c.tap_img2; p.swc = c.swc; p.w16 = c.w16; p.bog = c.bog;
  p.w_img = c.w_img; p.racc = c.racc; p.rowsum = c.rowsum; p.colsum = c.colsum; p.st_q = c.st_q;
  p.racc_tmap = *reinterpret_cast<const CUtensorMap*>(c.racc_tmap);
  const int npairs = (p.ntiles + 1) / 2;
  const dim3 grid(2 * std::min(ctx().sm_count / 2, npairs));
  if (c.slope2 <= 1.f) launch_k(k_dconv_mma2<true>, grid, dim3(kThreadsD), kSmemBytes, st, true, p);
  else launch_k(k_dconv_mma2<false>, grid, dim3(kThreadsD), kSmemBytes, st, true, p);
}

}  // namespace septfa
