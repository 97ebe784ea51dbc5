// K1+K2 with the mel projection on the 5th-generation tensor cores (tcgen05), n_fft = 512.
//
// Same operator as stft_mel.cu (the librosa chain under script/mfcc.py:387: centre-padded frames, periodic
// Hann, rFFT, |X|^2, Slaney mel, 10*log10, per-clip max), different execution model for the projection:
//
//   D[128 frames x n_mels] = P[128 x 272 bins] . W^T            (per block of 128 consecutive frames of a clip)
//
// issued as tcgen05.mma.cta_group::1.kind::f16 with BF16 operand pairs and FP32 accumulation in tensor memory:
//   P = b1 + b2   (b1 = the fp32 power rounded to bf16, b2 = the top 16 bits of the exact remainder),
//   W = w1 + w2   (round-to-nearest bf16 pair, built on the host),
//   D1 = b1.w1,  D2 = b1.w2 + b2.w1  (the large and the small terms in separate accumulator columns; b2.w2 is
//   below 2^-17 of the result), log-mel from D1 + D2.  bf16 keeps fp32's exponent range, so no per-frame scale is
//   needed although the power spectrum of a frame spans many decades; the relative error of a mel power is below
//   3e-5 (host emulation: tests/test_host.py; GPU bound: tests/test_gpu_parity.py, north_star 1e-4).
//
// One persistent 512-thread CTA per SM (16 warps; all 512 TMEM columns), organised as four independent 4-warp groups
// (see the kernel's own comment); bands [0, n_act) with at least one FFT bin (n_act rounded up to 16 <= 112):
//  * tile = 64 frames = one pass of the register FFT (32 half-warp groups x 2 frames, fft_regs.cuh / stft_core.cuh
//    exactly as in stft_mel.cu), PCM span by TMA; two tiles make one block of 128 frames = the M of the MMA;
//  * the split step leaves each group's two power rows ([frame][bin], fp32) in the group's OWN exchange buffer,
//    so the staging costs no shared memory beyond what the FFT needs anyway;
//  * transfer: every warp moves 16 frames x 1/4 of the bins from the rows into the A operand in tensor memory
//    with tcgen05.st.16x32bx2 (16 TMEM lanes per instruction: tile j of a block owns lanes 16 j .. 16 j + 15 of
//    every 32-lane quarter, so all 16 warps take part in every tile -- the 32-lane shape would leave half of them
//    idle; addressing and packing order checked by tools/ubench/tmem_st16.cu), splitting b1 / b2 on the way
//    (one integer add, one AND, half a packed subtract and one byte permute per bin);
//  * after the second tile the last warp to finish issues the 34 MMAs (17 K slabs x {N = 2 nb against [w1 | w2], N = nb against
//    w1}) and commits to an mbarrier; they run underneath the next tile's transform;
//  * epilogue (before the next block's first transfer): tcgen05.ld of D1, D2 (lane = frame), log, coalesced stores
//    along time, warp-shuffle max -> atomicMax per clip.
#include <cuda_bf16.h>

#include <cfloat>
#include <cstdint>
#include <cstring>
#include <vector>

#include "mmf_internal.h"
#include "stft_core.cuh"

namespace mmf {

namespace {

constexpr int kNfft = 512;
constexpr int kTcThreads = 512;
constexpr int kTcSlots = kTcThreads / 16;  // half-warp groups, two frames each
constexpr int kTcTF = 2 * kTcSlots;        // frames per tile (64)
constexpr int kTcBlock = 2 * kTcTF;        // frames per MMA block (128)
constexpr int kTcKP = 272;                 // bins padded to whole K = 16 slabs (257 -> 17 slabs)
constexpr int kTcSlabs = kTcKP / 16;
constexpr int kTcACols = kTcKP / 2;        // TMEM columns of one A operand (two bf16 per column)
// exchange buffer of a group, in 8-byte elements.  It also holds the group's two power rows after the split step:
// row A at float 0, row B at float 276, both shifted by 12 floats in odd groups.  With 274 elements (548 floats)
// per group the 32-bit row stores of the two groups of a warp fall on disjoint banks (548 + 12 = 16 mod 32) and
// the 128-bit row loads of eight consecutive frames on eight distinct 16-byte bank groups
// ((137 g + 69 parity + 3 (g & 1)) mod 8 is a permutation over four consecutive groups x two parities).
constexpr int kTcXS = 274;
constexpr int kTcRowB = 276;
constexpr int kTcOddShift = 12;
constexpr int kBox = 256;

__device__ __forceinline__ uint32_t tc_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void tc_mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(tc_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void tc_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(tc_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tc_mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "MMFTC_WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra MMFTC_DONE_%=;\n"
      "bra MMFTC_WAIT_%=;\n"
      "MMFTC_DONE_%=:\n"
      "}\n" ::"r"(tc_smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void tc_tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
          tc_smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(tc_smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ int tc_float_key(float f) {
  const int b = __float_as_int(f);
  return b >= 0 ? b : b ^ 0x7FFFFFFF;
}
__device__ __forceinline__ float tc_log2(float x) {
  float r;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ c2 tc_shfl(c2 v, int src) {
  const float xa = __shfl_sync(0xffffffffu, plo(v.x), src), xb = __shfl_sync(0xffffffffu, phi(v.x), src);
  const float ya = __shfl_sync(0xffffffffu, plo(v.y), src), yb = __shfl_sync(0xffffffffu, phi(v.y), src);
  return CxTraits<c2>::make(pmake(xa, xb), pmake(ya, yb));
}
__device__ __forceinline__ uint64_t tc_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
  uint64_t d = (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo >> 4) & 0x3FFFu) << 32;
  d |= 1ull << 46;
  return d;
}
// A from tensor memory (lane = frame, column j = bins 2j, 2j + 1 as bf16), B from shared memory, bf16 -> fp32
__device__ __forceinline__ void tc_mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, {%5, %5, %5, %5}, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(acc), "r"(0u)
      : "memory");
}
__device__ __forceinline__ void tc_tmem_ld4(uint32_t taddr, float* v) {
  uint32_t* u = reinterpret_cast<uint32_t*>(v);
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];"
               : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3])
               : "r"(taddr)
               : "memory");
}
// 16 TMEM lanes: threads 0-15 write columns [c, c + 16) of lanes base + t, threads 16-31 columns [c + 16, c + 32)
// of lanes base + t - 16
__device__ __forceinline__ void tc_tmem_st16x16(uint32_t taddr, const uint32_t* v) {
  asm volatile(
      "tcgen05.st.sync.aligned.16x32bx2.x16.b32 [%0], 16, {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]),
      "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
__device__ __forceinline__ void tc_tmem_st16x1(uint32_t taddr, uint32_t v) {
  asm volatile("tcgen05.st.sync.aligned.16x32bx2.x1.b32 [%0], 1, {%1};" ::"r"(taddr), "r"(v) : "memory");
}

// where the split step puts |X[k]|^2 of the group's two frames: one fp32 row per frame
struct SlotRows {
  float* a;
  float* b;
  __device__ __forceinline__ void put(int k, int, pk p) const {
    a[k] = plo(p);
    b[k] = phi(p);
  }
};

}  // namespace

struct StftTcArgs {
  const float* pcm;
  long n_samples;
  long clip_stride;
  int use_tma;              // 0: plain coalesced span loads (base or row pitch not 16-byte aligned)
  int span_floats;
  unsigned n_blocks;        // blocks of 128 frames over all clips
  unsigned blocks_per_clip;
  int T;
  int hop;
  int span_alloc;           // floats of a group's PCM span (16 frames of a tile), whole TMA boxes
  int lead;
  int vec_ok;
  int win_lo, win_hi;       // 32-sample groups [win_lo, win_hi) of the zero-padded window that are not all zero
  int n_mels;
  int n_act;                // bands [0, n_act) can be non-zero (the operand table covers them); [n_act, n_mels) are empty
  float amin;
  float preemph;
  const float* window;      // [512]
  const float2* tw1;        // [256]
  const uint16_t* wtab;     // bf16 [2 nb rows (w1 bands, then w2 bands) x 272] canonical K-major
  float* logmel;
  int* clipmax;
  int pitch;                // frames per log-mel row (T; the longest clip's T in a variable-length batch)
  // variable-length batch (null: every clip has n_samples samples and T frames): samples and frames of each clip,
  // and the first block of each clip over the blocks of all clips (vl_first[n_clips] = n_blocks)
  const long* vl_len;
  const int* vl_T;
  const unsigned* vl_first;
  int vl_clips;
};

// NBQ = bands per epilogue warp = nb / 4 (nb = the non-empty bands n_act rounded up to 16)
//
// Thread organisation.  Warp w = 4 cg + q.  The four warps with the same q (they share an SM sub-partition and,
// by the hardware's rule, the TMEM lane quarter q) form a GROUP: per tile the group transforms frames
// 16 q .. 16 q + 15 (eight half-warp frame pairs), transfers exactly those frames into lanes of quarter q, and
// later reads them back from D.  Everything a group waits for inside a tile is produced by the group itself, so
// its two barriers per tile are 128-thread named barriers and its PCM span has its own buffer and mbarrier: the
// four groups drift apart, one sub-partition's shared-memory phase running under the others' arithmetic (a
// deliberate start stagger of up to 4000 cycles between the groups measured no different: DESIGN.md section 6a).
// The only cross-group step is the MMA of a block: the last of the 16 warps to finish the block's transfers
// issues it (nobody waits), and every warp picks the result up one transform later.
// FAST160 = the bench / speech configuration (hop 160, TMA loader, no pre-emphasis) with the other load variants
// compiled out: the tile loop loses four code paths and their run-time predicates.
// VL = a variable-length batch (StftTcArgs::vl_*); compiled out of the equal-length instantiations.
template <int NBQ, bool FAST160, bool VL>
__global__ void __launch_bounds__(kTcThreads, 1)
    stft_mel_tc_kernel(const __grid_constant__ CUtensorMap tmap, const StftTcArgs p) {
  using C = FftCfg<kNfft>;
  using V = c2;
  constexpr int NB = 4 * NBQ;
  constexpr uint32_t kDCol = 2 * kTcACols;  // D1 at kDCol, D2 at kDCol + NB
  static_assert(2 * kTcACols + 2 * NB <= 512, "A (b1, b2) and D (D1, D2) must fit the 512 TMEM columns");
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  // hop 160 without pre-emphasis: 15 * 160 + 512 + 3 samples -> 3072 floats per group span, a compile-time constant
  // in the fast instantiation (every shared-memory offset below then folds into an immediate)
  const int span_alloc = FAST160 ? 3072 : p.span_alloc;
  float* s_span = reinterpret_cast<float*>(smem_raw);                           // [4][span_alloc]
  pk* s_xb = reinterpret_cast<pk*>(s_span + 4 * span_alloc);                    // [32][kTcXS]
  uint16_t* s_w = reinterpret_cast<uint16_t*>(s_xb + kTcSlots * kTcXS);         // [2 NB x 272] bf16
  c2* s_tw1 = reinterpret_cast<c2*>(s_w + 2 * NB * kTcKP);                      // [256]
  float2* s_win = reinterpret_cast<float2*>(s_tw1 + C::TW1);                    // [256] half-scaled window pairs
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_win + C::M);                  // [0..3] TMA of group q, [4] MMA
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_bar + 5);
  unsigned* s_cnt = s_tmem + 1;                                                 // warps that finished a block's transfers

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int tau = tid & 15;
  const int q = warp & 3, cg = warp >> 2, hw = lane >> 4;

  for (int i = tid; i < 2 * NB * kTcKP * 2 / 16; i += kTcThreads)
    reinterpret_cast<uint4*>(s_w)[i] = reinterpret_cast<const uint4*>(p.wtab)[i];
  for (int i = tid; i < C::TW1; i += kTcThreads) s_tw1[i] = make_tw<V>(p.tw1[i]);
  for (int i = tid; i < C::M; i += kTcThreads) {
    const float2 w = *reinterpret_cast<const float2*>(p.window + 2 * i);
    s_win[i] = make_float2(0.5f * w.x, 0.5f * w.y);  // the 1/2 of the real-FFT split step
  }
  c2 wtau;
  {
    float2 w;
    sincospif(-2.0f * (float)tau / (float)kNfft, &w.y, &w.x);
    wtau = make_tw<V>(w);
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc_smem_u32(s_tmem)), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (tid == 0) {
    for (int i = 0; i < 5; ++i) tc_mbar_init(&s_bar[i], 1);
    *s_cnt = 0;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // the operand table is read by the tensor core
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = *s_tmem;

  // ---- roles
  // transform: half-warp (cg, hw) of group q owns frames 4 cg + 2 hw, + 1 of the group's 16; exchange buffer
  // 8 q + 2 cg + hw (a group's buffers are consecutive: the row loads below rely on it, see kTcXS)
  const int xbi = 8 * q + 2 * cg + hw;
  pk* xb = s_xb + xbi * kTcXS;
  float* row_a = reinterpret_cast<float*>(xb) + (xbi & 1) * kTcOddShift;
  const SlotRows rows{row_a, row_a + kTcRowB};
  const int f_own = 4 * cg + 2 * hw;  // first of this half-warp's two frames within the group
  // transfer: warp cg of group q moves the group's 16 frames (lane & 15), bins [64 cg, 64 cg + 64) (lanes 0-15 the
  // first 32 of them, lanes 16-31 the second 32) plus two of the eight tail columns (bins 256 ..)
  const int tfr = lane & 15;
  const int tbi = 8 * q + (tfr >> 1);
  const float* trow = reinterpret_cast<const float*>(s_xb + tbi * kTcXS) + (tbi & 1) * kTcOddShift + (tfr & 1) * kTcRowB;
  const float* tsrc = trow + 64 * cg + 32 * hw;
  const uint32_t lane_q = (uint32_t)(32 * q) << 16;
  float* span = s_span + q * span_alloc;
  uint64_t* bar_tma = &s_bar[q];
  uint64_t* bar_mma = &s_bar[4];
  auto group_sync = [&]() { asm volatile("bar.sync %0, 128;" ::"r"(q + 1) : "memory"); };

  const uint32_t idesc2 = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)((2 * NB) >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
  const uint32_t idesc1 = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(NB >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
  const uint64_t wdesc = tc_desc(tc_smem_u32(s_w), 128, (uint32_t)(kTcKP / 8) * 128);

  const int hop = FAST160 ? 160 : p.hop, lead = FAST160 ? 0 : p.lead;
  const uint32_t n_boxes = (uint32_t)span_alloc / kBox;
  auto clip_len = [&](int clip) -> long { return VL ? p.vl_len[clip] : p.n_samples; };
  auto clip_T = [&](int clip) -> int { return VL ? p.vl_T[clip] : p.T; };

  // block sequence of this CTA: blocks blockIdx.x, + gridDim.x, ...; 1 or 2 tiles of 64 frames per block
  auto block_pos = [&](unsigned blk, int& clip, int& t0) {
    if (VL) {  // the last clip whose first block is <= blk (clips without blocks are skipped over)
      int lo = 0, hi = p.vl_clips - 1;
      while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (p.vl_first[mid] <= blk) lo = mid;
        else hi = mid - 1;
      }
      clip = lo;
      t0 = (int)(blk - p.vl_first[lo]) * kTcBlock;
      return;
    }
    clip = (int)(blk / p.blocks_per_clip);
    t0 = (int)(blk - (unsigned)clip * p.blocks_per_clip) * kTcBlock;
  };
  // variable-length batch: the TMA fills the span from the padded buffer, whose samples at and past the clip's end
  // must read as zero -- overwrite them before the group's frames load (the group syncs only when it wrote)
  auto zero_tail = [&](int clip, int t0) {
    if (!VL) return;
    const long g0 = (long)(((t0 + 16 * q) * hop - kNfft / 2 - lead) & ~3);
    const long from = clip_len(clip) - g0;
    if (from >= span_alloc) return;
    for (long i = max(0L, from) + 32 * cg + lane; i < span_alloc; i += 128) span[i] = 0.0f;
    group_sync();
  };
  // warp cg == 0 of the group: the PCM span of the group's 16 frames of tile t0, one 1 KB box per TMA
  auto issue_span = [&](int clip, int t0) {
    const int g0 = ((t0 + 16 * q) * hop - kNfft / 2 - lead) & ~3;  // 16-byte aligned start (remainder: `shift`)
    if (lane == 0) {
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      tc_mbar_expect_tx(bar_tma, (uint32_t)span_alloc * 4u);
    }
    __syncwarp();
    for (uint32_t bx = lane; bx < n_boxes; bx += 32) tc_tma_load_2d(span + bx * kBox, &tmap, g0 + (int)bx * kBox, clip, bar_tma);
  };
  // plain loader (no TMA): same span, same zero fill outside the clip
  auto fill_span = [&](int clip, int t0) {
    const long g0 = (long)(((t0 + 16 * q) * hop - kNfft / 2 - lead) & ~3);
    const float* src = p.pcm + (size_t)clip * p.clip_stride;
    const long len = clip_len(clip);
    for (int i = 32 * cg + lane; i < p.span_floats; i += 128) {
      const long n = g0 + i;
      span[i] = (n >= 0 && n < len) ? __ldg(src + n) : 0.0f;
    }
    group_sync();
  };
  auto issue_mma = [&]() {  // one thread: D1 | D2 = b1 . [w1 | w2], D2 += b2 . w1 over the 17 K slabs
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
    for (int s = 0; s < kTcSlabs; ++s) {
      tc_mma_ts(tmem + kDCol, tmem + 8 * s, wdesc + 16 * s, idesc2, s > 0 ? 1u : 0u);
      tc_mma_ts(tmem + kDCol + NB, tmem + kTcACols + 8 * s, wdesc + 16 * s, idesc1, 1u);
    }
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(tc_smem_u32(bar_mma)) : "memory");
  };
  // D (tensor memory) -> log-mel rows of block (clip, t0): warp (q, cg) handles lanes 32 q .. 32 q + 31 (frames
  // t0 + 64 (lane / 16) + 16 q + lane % 16) and bands [NBQ cg, NBQ cg + NBQ)
  auto epilogue = [&](int clip, int t0) {
    float d1[NBQ], d2[NBQ];
#pragma unroll
    for (int i = 0; i < NBQ; i += 4) {
      tc_tmem_ld4(tmem + lane_q + kDCol + NBQ * cg + i, d1 + i);
      tc_tmem_ld4(tmem + lane_q + kDCol + NB + NBQ * cg + i, d2 + i);
    }
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    const int t = t0 + kTcTF * hw + 16 * q + (lane & 15);
    const int pitch = p.pitch;
    float mx = -FLT_MAX;
    if (t < clip_T(clip)) {
      float* dst = p.logmel + ((size_t)clip * p.n_mels + NBQ * cg) * pitch + t;
      const int n_here = min(NBQ, p.n_act - NBQ * cg);  // bands of this warp that exist
      const float amin = p.amin;
#pragma unroll
      for (int i = 0; i < NBQ; ++i) {
        if (i < n_here) {
          // 10*log10(x) = 10*log10(2) * log2(x); MUFU.LG2 is within 1e-6 dB here (x >= amin, never denormal)
          const float db = 3.01029995663981195f * tc_log2(fmaxf(amin, d1[i] + d2[i]));
          *dst = db;
          dst += pitch;
          mx = fmaxf(mx, db);
        }
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if (lane == 0 && mx > -FLT_MAX) atomicMax(p.clipmax + clip, tc_float_key(mx));
  };

  unsigned blk = blockIdx.x;
  int clip = 0, t0b = 0;
  // (clip, first frame) of this CTA's next block advance by gridDim.x blocks without dividing again
  const unsigned step_q = gridDim.x / p.blocks_per_clip, step_r = gridDim.x - step_q * p.blocks_per_clip;
  unsigned bin = 0;  // block index within the clip
  if (blk < p.n_blocks) {
    block_pos(blk, clip, t0b);
    bin = (unsigned)t0b / kTcBlock;
    if ((FAST160 || p.use_tma) && cg == 0) issue_span(clip, t0b);
  }
  uint32_t tma_par = 0, mma_par = 0;
  bool have_prev = false;  // a block whose MMAs are issued (or about to be) and whose D has not been written out yet
  int pclip = 0, pt0 = 0;

  while (blk < p.n_blocks) {
    const int n_tiles = (t0b + kTcTF < clip_T(clip)) ? 2 : 1;
    const unsigned nblk = blk + gridDim.x;
    int nclip = clip + (int)step_q;
    unsigned nbin = bin + step_r;
    if (nbin >= p.blocks_per_clip) {
      nbin -= p.blocks_per_clip;
      ++nclip;
    }
    int nt0b = (int)nbin * kTcBlock;
    if (VL && nblk < p.n_blocks) block_pos(nblk, nclip, nt0b);
    for (int j = 0; j < n_tiles; ++j) {
      const int t0 = t0b + kTcTF * j;
      const int g_first = (t0 + 16 * q) * hop - kNfft / 2 - lead;
      const int shift = g_first - (g_first & ~3);
      // ---------------- load phase: two frames per half-warp into registers
      V v[16];
      {
        float2 wreg[16];
#pragma unroll
        for (int n2 = 0; n2 < 16; ++n2) wreg[n2] = s_win[tau + C::TPF * n2];
        const int off = shift + lead + f_own * hop;
        if constexpr (FAST160) {
          tc_mbar_wait(bar_tma, tma_par);
          tma_par ^= 1u;
          zero_tail(clip, t0);
          // (shift == 0: the spans start 16-byte aligned.)  The 25 ms window of speech front ends (400 of 512) as
          // compile-time bounds: the 21 load predicates of the generic form disappear
          if (p.win_lo == 1 && p.win_hi == 15)
            ph_load_shared<kNfft, 5, true>(v, span, off, tau, wreg, 1, 15);
          else
            ph_load_shared<kNfft, 5, true>(v, span, off, tau, wreg, p.win_lo, p.win_hi);
        } else {
          if (p.use_tma) {
            tc_mbar_wait(bar_tma, tma_par);
            tma_par ^= 1u;
            zero_tail(clip, t0);
          } else {
            fill_span(clip, t0);  // (the previous tile's frames left the buffer before its first barrier)
          }
          if (p.preemph != 0.0f) {
            const long n_valid = clip_len(clip) - ((long)(t0 + 16 * q + f_own) * hop - kNfft / 2);
            ph_load_pre<kNfft>(v, span, off, hop, tau, wreg, p.preemph, n_valid);
          } else if (hop == 160 && !(shift & 1)) {
            ph_load_shared<kNfft, 5, true>(v, span, off, tau, wreg, p.win_lo, p.win_hi);
          } else if (hop == 128 && !(shift & 1)) {
            ph_load_shared<kNfft, 4, true>(v, span, off, tau, wreg, p.win_lo, p.win_hi);
          } else if (hop == 256 && !(shift & 1)) {
            ph_load_shared<kNfft, 8, true>(v, span, off, tau, wreg, p.win_lo, p.win_hi);
          } else if (p.vec_ok && !(shift & 1)) {
            ph_load<kNfft, true>(v, span, off, hop, tau, wreg);
          } else {
            ph_load<kNfft, false>(v, span, off, hop, tau, wreg);
          }
        }
      }
      // the group's frames sit in registers: its span buffer is free, and its previous transfer (which read the
      // group's exchange buffers) is complete
      group_sync();
      if ((FAST160 || p.use_tma) && cg == 0) {
        if (j + 1 < n_tiles)
          issue_span(clip, t0 + kTcTF);
        else if (nblk < p.n_blocks)
          issue_span(nclip, nt0b);
      }
      // ---------------- transform (as stft_mel.cu, two frames per half-warp on packed FP32)
      ph_pass1<kNfft>(v, s_tw1, tau);
      __syncwarp();
      ph_x1_write<kNfft, 1>(v, xb, tau);
      __syncwarp();
      ph_x1_read<kNfft, 1>(v, xb, tau);
      __syncwarp();
      ph_x1_write<kNfft, 2>(v, xb, tau);
      __syncwarp();
      ph_x1_read<kNfft, 2>(v, xb, tau);
      ph_pass2<kNfft>(v, s_tw1 /* unused: R3 == 1 */, tau);
      {
        // partner lane holds Z[M - k]: lane (16 - tau) & 15 of the same half-warp, register 15 - r
        const int src = ((16 - tau) & 15) | (lane & 16);
        V bpart[8];
#pragma unroll
        for (int r = 0; r < 8; ++r) {
          const V sh = tc_shfl(v[15 - r], src);
          bpart[r] = (tau == 0) ? v[(16 - r) & 15] : sh;
        }
        __syncwarp();  // the half-warp's exchange reads are done: its buffer now takes the two power rows
        ph_split_regs512_to(v, bpart, rows, 0, tau, wtau);
      }
      group_sync();  // the group's power rows are complete
      // ---------------- previous block: D -> log-mel (its MMAs ran underneath this tile's transform)
      if (j == 0 && have_prev) {
        tc_mbar_wait(bar_mma, mma_par);
        mma_par ^= 1u;
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        epilogue(pclip, pt0);
        have_prev = false;
      }
      // ---------------- transfer: rows -> b1 / b2 -> A operand in tensor memory (lanes 16 j .. 16 j + 15 of quarter q)
      {
        const uint32_t a_lane = tmem + lane_q + ((uint32_t)(16 * j) << 16);
        uint32_t b1[16], b2[16];
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const float4 x = *reinterpret_cast<const float4*>(tsrc + 4 * c);
          const float xs[4] = {x.x, x.y, x.z, x.w};
          // b1 = the power rounded to bf16 (half an ulp added to the bits, top half kept), b2 = the top half of the
          // exact, signed remainder.  Rounding b1 instead of truncating it halves |b2| and makes the neglected
          // b2.w2 term and b2's own truncation zero-mean: worst mel-power error 5.0e-5 -> 2.9e-5 on the emulation
          // (tests/test_host.py::test_bf16_pair_mel_projection_accuracy) for one more integer add per bin
          uint32_t us[4];
          float ts[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            us[e] = __float_as_uint(xs[e]) + 0x8000u;
            ts[e] = __uint_as_float(us[e] & 0xffff0000u);
          }
          // exact remainders, two per packed subtract
          const pk r01 = ssub(pmake(xs[0], xs[1]), pmake(ts[0], ts[1])), r23 = ssub(pmake(xs[2], xs[3]), pmake(ts[2], ts[3]));
          const float rs[4] = {plo(r01), phi(r01), plo(r23), phi(r23)};
          b1[2 * c] = __byte_perm(us[0], us[1], 0x7632);
          b1[2 * c + 1] = __byte_perm(us[2], us[3], 0x7632);
          b2[2 * c] = __byte_perm(__float_as_uint(rs[0]), __float_as_uint(rs[1]), 0x7632);
          b2[2 * c + 1] = __byte_perm(__float_as_uint(rs[2]), __float_as_uint(rs[3]), 0x7632);
        }
        tc_tmem_st16x16(a_lane + 32 * cg, b1);
        tc_tmem_st16x16(a_lane + kTcACols + 32 * cg, b2);
        // tail columns 128 .. 135 (bins 256 .. 271): only bin 256 exists, the rest of the K padding is zero
        uint32_t t1 = 0, t2 = 0;
        if (cg == 0 && hw == 0) {
          const float x = trow[256];
          const uint32_t u = __float_as_uint(x) + 0x8000u;
          const float r = x - __uint_as_float(u & 0xffff0000u);
          t1 = u >> 16;
          t2 = __float_as_uint(r) >> 16;
        }
        tc_tmem_st16x1(a_lane + 128 + 2 * cg, t1);
        tc_tmem_st16x1(a_lane + kTcACols + 128 + 2 * cg, t2);
        // (no wait here: the stores only have to be complete when this warp reports the block below)
      }
    }
    // ---------------- the block's A operand is complete once all 16 warps have been here: the last one issues the MMAs
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncwarp();
    if (lane == 0) {
      __threadfence_block();
      const unsigned arrived = atomicAdd(s_cnt, 1u);
      if ((arrived & 15u) == 15u) {
        __threadfence_block();
        issue_mma();
      }
    }
    __syncwarp();
    have_prev = true;
    pclip = clip;
    pt0 = t0b;
    blk = nblk;
    clip = nclip;
    bin = nbin;
    t0b = nt0b;
  }
  // ---------------- drain: epilogue of the last block
  if (have_prev) {
    tc_mbar_wait(bar_mma, mma_par);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    epilogue(pclip, pt0);
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512) : "memory");
}

// Bands without a single FFT bin (fmax above the Nyquist frequency: the reference's GUI default asks for 10 kHz at a
// 10 kHz sampling rate, script/main.py:739) are not part of the GEMM: mel power 0 -> the amin floor, as librosa gives.
// vT (variable-length batch, else null): frames of each clip, 0 for a clip this launch does not cover.
__global__ void mel_empty_bands_kernel(float* __restrict__ logmel, int* __restrict__ clipmax, int T, int pitch,
                                       const int* __restrict__ vT, int n_mels, int n_act, float amin) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int clip = blockIdx.y;
  if (vT) {
    T = vT[clip];
    if (T == 0) return;
  }
  const float db0 = 3.01029995663981195f * tc_log2(fmaxf(amin, 0.0f));
  if (t < T)
    for (int b = n_act; b < n_mels; ++b) logmel[((size_t)clip * n_mels + b) * pitch + t] = db0;
  if (blockIdx.x == 0 && threadIdx.x == 0) atomicMax(clipmax + clip, tc_float_key(db0));
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------

static int tc_nb(int n_mels) { return (n_mels + 15) / 16 * 16; }

static size_t tc_smem_bytes(int span_alloc, int nb) {
  using C = FftCfg<kNfft>;
  return (size_t)4 * span_alloc * 4 + (size_t)kTcSlots * kTcXS * 8 + (size_t)2 * nb * kTcKP * 2 +
         (size_t)C::TW1 * sizeof(c2) + (size_t)C::M * 8 + 5 * 8 + 16;
}

// floats of the PCM span of one group (16 frames), whole TMA boxes
int stft_mel_tc_span_alloc(int hop, int lead) { return (15 * hop + kNfft + lead + 3 + kBox - 1) / kBox * kBox; }

// bands [0, n_act) have at least one non-zero weight somewhere (trailing bands above the Nyquist frequency are empty)
int stft_mel_tc_active_bands(const std::vector<float>& mel, int n_mels, int F) {
  int n_act = 1;
  for (int m = 0; m < n_mels; ++m)
    for (int k = 0; k < F; ++k)
      if (mel[(size_t)m * F + k] != 0.0f) n_act = m + 1;
  return n_act;
}

// n_fft = 512 on the packed two-frame transform; the non-empty bands (rounded up to 16) must leave A (272 columns)
// and D (2 nb columns) inside the 512 TMEM columns, and the tile spans + tables inside one SM's shared memory
bool stft_mel_tc_supported(int n_fft, int n_act, int hop, int lead, int packed) {
  if (n_fft != kNfft || !packed || n_act < 1 || tc_nb(n_act) > 112 || hop < 1) return false;
  return tc_smem_bytes(stft_mel_tc_span_alloc(hop, lead), tc_nb(n_act)) <= 227 * 1024;
}

static uint16_t bf16_rn_bits(float f) {
  uint32_t u;
  std::memcpy(&u, &f, 4);
  u += 0x7fffu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}
static float bf16_to_float(uint16_t b) {
  const uint32_t u = (uint32_t)b << 16;
  float f;
  std::memcpy(&f, &u, 4);
  return f;
}

// mel: dense [n_mels][F] filterbank (host_mel_dense).  tab: 2 nb rows x 272 bf16, canonical no-swizzle K-major
// ((row / 8) * (272 / 8) + k / 8) * 64 + (row % 8) * 8 + k % 8; rows [0, nb) = w1 of band row, rows [nb, 2 nb) = w2
void stft_mel_tc_table(const std::vector<float>& mel, int n_mels, int F, std::vector<uint16_t>& tab) {
  n_mels = stft_mel_tc_active_bands(mel, n_mels, F);  // rows of the table = non-empty bands
  const int nb = tc_nb(n_mels);
  tab.assign((size_t)2 * nb * kTcKP, 0);
  auto idx = [&](int row, int k) { return ((size_t)(row / 8) * (kTcKP / 8) + k / 8) * 64 + (row % 8) * 8 + k % 8; };
  for (int m = 0; m < n_mels; ++m)
    for (int k = 0; k < F && k < kTcKP; ++k) {
      const float w = mel[(size_t)m * F + k];
      const uint16_t w1 = bf16_rn_bits(w);
      const uint16_t w2 = bf16_rn_bits(w - bf16_to_float(w1));
      tab[idx(m, k)] = w1;
      tab[idx(nb + m, k)] = w2;
    }
}

cudaError_t stft_mel_tc_launch(const CUtensorMap& tmap, int use_tma, const float* pcm, long n_clips, long n_samples,
                               long clip_stride, int T, int hop,
                               int lead, int n_mels, int n_act, float amin, float preemph, const float* window, int win_lo,
                               int win_hi, const float2* tw1, const void* wtab, float* logmel, int* clipmax,
                               int sm_count, cudaStream_t st, const Varlen* vl) {
  StftTcArgs a{};
  a.win_lo = win_lo;
  a.win_hi = win_hi;
  const long bpc = (T + kTcBlock - 1) / kTcBlock;
  if (bpc * n_clips > 0x7fffffffL) return cudaErrorInvalidValue;
  a.pitch = T;
  if (vl) {
    a.vl_len = vl->len;
    a.vl_T = vl->T;
    a.vl_first = vl->first;
    a.vl_clips = (int)n_clips;
    a.pitch = vl->pitch;
  }
  a.pcm = pcm;
  a.n_samples = n_samples;
  a.clip_stride = clip_stride;
  a.use_tma = use_tma;
  a.span_floats = 15 * hop + kNfft + lead + 3;
  a.blocks_per_clip = (unsigned)bpc;
  a.n_blocks = vl ? (unsigned)vl->n_units : (unsigned)(bpc * n_clips);
  a.T = T;
  a.hop = hop;
  a.span_alloc = stft_mel_tc_span_alloc(hop, lead);
  a.lead = lead;
  a.vec_ok = (hop % 2 == 0) ? 1 : 0;
  a.n_mels = n_mels;
  a.n_act = n_act;
  a.amin = amin;
  a.preemph = preemph;
  a.window = window;
  a.tw1 = tw1;
  a.wtab = reinterpret_cast<const uint16_t*>(wtab);
  a.logmel = logmel;
  a.clipmax = clipmax;
  const int nb = tc_nb(n_act);
  const size_t smem = tc_smem_bytes(a.span_alloc, nb);
  const unsigned grid = (unsigned)std::min<long>((long)a.n_blocks, (long)sm_count);
  const bool fast160 = hop == 160 && use_tma && preemph == 0.0f && lead == 0 && a.span_alloc == 3072;
#define MMF_TCMEL_LAUNCH(NBQ, F, V)                                \
  {                                                                \
    auto kfn = stft_mel_tc_kernel<NBQ, F, V>;                      \
    MMF_SMEM_ONCE(kfn, 227 * 1024);                                \
    kfn<<<grid, kTcThreads, smem, st>>>(tmap, a);                  \
  }
#define MMF_TCMEL_CASE(NBQ)                                        \
  case NBQ: {                                                      \
    if (fast160) {                                                 \
      if (vl) MMF_TCMEL_LAUNCH(NBQ, true, true)                    \
      else MMF_TCMEL_LAUNCH(NBQ, true, false)                      \
    } else {                                                       \
      if (vl) MMF_TCMEL_LAUNCH(NBQ, false, true)                   \
      else MMF_TCMEL_LAUNCH(NBQ, false, false)                     \
    }                                                              \
    break;                                                         \
  }
  switch (nb / 4) {
    MMF_TCMEL_CASE(4)
    MMF_TCMEL_CASE(8)
    MMF_TCMEL_CASE(12)
    MMF_TCMEL_CASE(16)
    MMF_TCMEL_CASE(20)
    MMF_TCMEL_CASE(24)
    MMF_TCMEL_CASE(28)
    default: return cudaErrorInvalidValue;
  }
#undef MMF_TCMEL_CASE
#undef MMF_TCMEL_LAUNCH
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess && n_act < n_mels) {
    for (long c0 = 0; c0 < n_clips && e == cudaSuccess; c0 += 65535) {
      const unsigned nc = (unsigned)std::min<long>(65535, n_clips - c0);
      mel_empty_bands_kernel<<<dim3((unsigned)((a.pitch + 255) / 256), nc), 256, 0, st>>>(
          logmel + (size_t)c0 * n_mels * a.pitch, clipmax + c0, T, a.pitch, vl ? vl->T + c0 : nullptr, n_mels, n_act,
          amin);
      count_launch();
      e = cudaGetLastError();
    }
  }
  return e;
}

}  // namespace mmf
