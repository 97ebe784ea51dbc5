// K1+K2: fused frame -> (pre-emphasis) -> Hann window -> real FFT -> |X|^2 ->
// Slaney mel projection -> 10*log10 -> per-clip max, for a batch of clips.
//
// Replaces the librosa chain invoked at script/mfcc.py:387 (stft, abs**2,
// filters.mel + einsum, power_to_db before the top_db clamp).
//
// Execution model (sm_100a):
//  * persistent CTAs (2 per SM x 256 threads; 1 x 512 where only one fits), each
//    looping over tiles of TF consecutive frames of one clip (TF = 32 when it fits);
//  * the PCM span of a tile ((TF-1)*hop + n_fft samples, hop windows overlap) is
//    brought in once by TMA (cp.async.bulk.tensor, 1 KB boxes, mbarrier
//    completion); out-of-range coordinates are zero-filled by the TMA unit, which
//    *is* librosa's center=True / pad_mode='constant' padding, so no padded copy
//    of the audio ever exists.  With one span buffer the next tile's TMA is issued
//    as soon as every warp holds its frames in registers and streams in under the
//    transform and the mel projection;
//  * FFT data lives in registers, 16 complex points per thread -- by default of TWO
//    adjacent frames at once, packed for FADD2/FMUL2/FFMA2 (fft_regs.cuh) -- with
//    one shared-memory exchange between radix-16 passes; for n_fft = 512 the
//    real-FFT split step pairs bins with warp shuffles;
//  * the power tile stays in shared memory and is projected on the (sparse,
//    two-slopes-per-bin) mel filterbank by all warps, one frame per lane, band
//    groups balanced on the host (optionally on the tensor cores: mma.sync TF32 x3),
//    log'd and streamed out with coalesced stores; the 1 MB/clip power spectrum
//    never touches HBM unless the caller asks for it (mmf_stft_power).
#include <cfloat>
#include <cstdint>

#include "mmf_internal.h"
#include "stft_core.cuh"

namespace mmf {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "MMF_WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra MMF_DONE_%=;\n"
      "bra MMF_WAIT_%=;\n"
      "MMF_DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
          smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(smem_u32(bar))
      : "memory");
}

// monotone float -> int key so that atomicMax(int) orders like float compare
__device__ __forceinline__ int float_key(float f) {
  int b = __float_as_int(f);
  return b >= 0 ? b : b ^ 0x7FFFFFFF;
}

// barrier over the TPF threads that transform one frame (pair): a warp-level sync when they
// share a warp, otherwise a named barrier of their own (ids 1..15; id 0 is __syncthreads)
template <int TPF>
__device__ __forceinline__ void frame_sync(int slot) {
  if constexpr (TPF <= 32) {
    __syncwarp();
  } else {
    asm volatile("bar.sync %0, %1;" ::"r"(slot + 1), "r"(TPF) : "memory");
  }
}

constexpr int kThreads = 256;
constexpr int kBox = 256;  // floats per TMA box (1 KB)
constexpr int kMaxWorkers = 256;  // mel band groups per CTA: 8 warps * (32 / TF), TF >= 1

// One thread queues the TMA boxes of a tile's PCM span.  Negative and
// past-the-end sample coordinates are zero-filled by the TMA unit.
template <int NFFT>
__device__ __forceinline__ void issue_span(const CUtensorMap* tmap, const StftArgs& p, int clip, int t0, float* dst,
                                           uint64_t* bar) {
  // TMA box start addresses must be 16-byte aligned: round the first sample down
  // to a multiple of 4 floats; the kernel adds the remainder to its frame offsets
  const int g0 = (t0 * p.hop - NFFT / 2 - p.lead) & ~3;
  // order earlier generic-proxy accesses of this buffer before the async-proxy writes
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  mbar_expect_tx(bar, (uint32_t)p.span_alloc * 4u);
  for (int bx = 0; bx < p.span_alloc / kBox; ++bx) tma_load_2d(dst + bx * kBox, tmap, g0 + bx * kBox, clip, bar);
}

// shuffle of a complex value from lane src (one shuffle per 32-bit half)
__device__ __forceinline__ float2 shfl_cx(float2 v, int src) {
  return make_float2(__shfl_sync(0xffffffffu, v.x, src), __shfl_sync(0xffffffffu, v.y, src));
}
__device__ __forceinline__ c2 shfl_cx(c2 v, int src) {
  const float xa = __shfl_sync(0xffffffffu, plo(v.x), src), xb = __shfl_sync(0xffffffffu, phi(v.x), src);
  const float ya = __shfl_sync(0xffffffffu, plo(v.y), src), yb = __shfl_sync(0xffffffffu, phi(v.y), src);
  return CxTraits<c2>::make(pmake(xa, xb), pmake(ya, yb));
}

// ---- tensor-core mel projection -------------------------------------------------
// D[frame][band] += A[frame][bin] * B[bin][band] with mma.sync m16n8k8 TF32, three MMAs per
// product (hi*hi + hi*lo + lo*hi, fp32 accumulate): single-pass TF32 fails the 1e-4 tolerance
// on mel power, the 3-term split is accurate to ~2^-21.
__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, "
      "{%0, %1, %2, %3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ float fast_log2(float x) {
  float r;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
constexpr int kMaxUnits = 16;  // (n-tile, m-tile) units per warp: n_mels <= 512 -> 64 n-tiles x 2 / 8 warps

// V = float2: one frame per thread group; V = c2: two adjacent frames per thread group on
// packed FP32 instructions (fft_regs.cuh)
// THREADS = 256: two CTAs per SM; THREADS = 512: one CTA per SM with twice the warps, for
// configurations (large n_fft) whose tiles leave room for only one CTA
// MG = true: power tile in the bin-pair layout (TilePairs) and the grouped mel walk (mel_groups);
// MG = false: [bin][frame] rows, sparse walk or mma.sync mel
template <int NFFT, typename V, int THREADS, bool MG>
__global__ void __launch_bounds__(THREADS, THREADS == 256 ? 2 : 1)
    stft_mel_kernel(const __grid_constant__ CUtensorMap tmap, const StftArgs p) {
  constexpr int kThreads = THREADS;  // (shadows the file-level default inside the kernel)
  using C = FftCfg<NFFT>;
  using TR = CxTraits<V>;
  using Tw = typename TR::Tw;
  using Xe = typename TR::Xe;
  constexpr int SLOTS = kThreads / C::TPF;      // thread groups (one or two frames each)
  constexpr int FPI = SLOTS * TR::kFrames;      // frames transformed per iteration
  extern __shared__ __align__(1024) unsigned char smem_raw[];

  // ---- shared memory carve-up (mirrors stft_smem_bytes() on the host)
  float* s_span = reinterpret_cast<float*>(smem_raw);                       // [span_bufs][span_alloc]
  float* s_ptile = s_span + p.span_bufs * p.span_alloc;                     // [pt_bufs][F*ppitch]
  // bin rows padded to the MMA K tile (rows layout) / bin-pair rows padded to whole 4-bin groups (pair
  // layout: ppitch counts 8-byte words); the pad rows stay zero
  constexpr int FP = MG ? 4 * ((C::F + 3) / 4) : ((C::F + 7) & ~7);
  Xe* s_xb = reinterpret_cast<Xe*>(s_ptile + ((p.pt_bufs * FP * p.ppitch + 3) & ~3));  // [SLOTS][XBUF]
  Tw* s_tw1 = reinterpret_cast<Tw*>(s_xb + SLOTS * C::XSTRIDE);                // [TW1]
  Tw* s_tw2 = s_tw1 + C::TW1;                                               // [TW2]
  float2* s_win = reinterpret_cast<float2*>(s_tw2 + C::TW2);                // [M] half-scaled window pairs
  // mel tables: sparse FP32 walk            | tensor cores
  //   s_w2  [F] (falling, rising) weights   |   s_bw    [n_pairs][32] B fragments (fp32, split on the fly)
  //   s_seg [n_mels + 2] segment starts     |   s_pk8   [n_pairs] k-tile of each pair
  //   s_mb  [kMaxWorkers + 2] band groups   |   s_npair [NT + 1] pair range of each n-tile
  //                                         |   s_tile  [NT] first band | bands << 16 of each n-tile
  //                                         |   s_units [8][kMaxUnits] (n | m << 8) work list per warp
  // grouped walk: s_mgw [2 * mg_n] float4 weights | s_mgseg [n_mels + 2] int2 | s_mgstep [n_mels + 3] int2 | s_mb
  float2* s_w2 = s_win + C::M;
  int* s_seg = reinterpret_cast<int*>(s_w2 + C::F);
  int* s_mb = MG ? reinterpret_cast<int*>(s_win + C::M) + 8 * p.mg_n + 2 * (p.n_mels + 2) + 2 * (p.n_mels + 3)
                 : s_seg + ((p.n_mels + 2 + 1) & ~1);
  float4* s_mgw = reinterpret_cast<float4*>(s_win + C::M);
  int2* s_mgseg = reinterpret_cast<int2*>(s_mgw + 2 * p.mg_n);
  int2* s_mgstep = s_mgseg + (p.n_mels + 2);
  float2* s_bw = s_win + C::M;
  int* s_pk8 = reinterpret_cast<int*>(s_bw + (size_t)p.mma_n_pairs * 32);
  int* s_npair = s_pk8 + p.mma_n_pairs;
  int* s_tile = s_npair + (p.mma_n_tiles + 1);
  int* s_units = s_tile + p.mma_n_tiles;
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(
      reinterpret_cast<unsigned char*>(s_win + C::M) + ((p.mel_tab_bytes + 15) & ~15));  // [2]

  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int tau = tid % C::TPF;
  const int slot = tid / C::TPF;

  for (int i = tid; i < C::TW1; i += kThreads) s_tw1[i] = make_tw<V>(p.tw1[i]);
  for (int i = tid; i < C::TW2; i += kThreads) s_tw2[i] = make_tw<V>(p.tw2[i]);
  if constexpr (MG) {
    for (int i = tid; i < 2 * p.mg_n; i += kThreads) s_mgw[i] = p.mg_w[i];
    for (int i = tid; i < p.n_mels + 2; i += kThreads) s_mgseg[i] = p.mg_seg[i];
    for (int i = tid; i < p.n_mels + 3; i += kThreads) s_mgstep[i] = p.mg_step[i];
    for (int i = tid; i < kMaxWorkers + 1; i += kThreads) s_mb[i] = p.band_split[i];
  } else if (p.mel_mma) {
    const int NT = p.mma_n_tiles;
    for (int i = tid; i < NT; i += kThreads) s_tile[i] = p.mma_tile[i];
    for (int i = tid; i < p.mma_n_pairs * 32; i += kThreads) s_bw[i] = p.mma_bw[i];
    for (int i = tid; i < p.mma_n_pairs; i += kThreads) s_pk8[i] = p.mma_pk8[i];
    for (int i = tid; i < NT + 1; i += kThreads) s_npair[i] = p.mma_npair[i];
    for (int i = tid; i < 8 * kMaxUnits; i += kThreads) s_units[i] = p.mma_units[i];
  } else {
    for (int i = tid; i < C::F; i += kThreads) s_w2[i] = p.w2[i];
    for (int i = tid; i < p.n_mels + 2; i += kThreads) s_seg[i] = p.seg_start[i];
    for (int i = tid; i < kMaxWorkers + 1; i += kThreads) s_mb[i] = p.band_split[i];
  }
  for (int i = tid; i < p.pt_bufs * FP * p.ppitch; i += kThreads) s_ptile[i] = 0.0f;  // incl. the K pad rows

  // Hann window pre-scaled by the 1/2 of the split step.  One frame per thread group: the
  // thread's 16 complex points stay in registers; two frames: registers are needed for the
  // second frame, so the window is staged in shared memory and re-read per iteration.
  constexpr bool kWinRegs = TR::kFrames == 1;
  for (int i = tid; i < C::M; i += kThreads) {
    const float2 w = *reinterpret_cast<const float2*>(p.window + 2 * i);
    s_win[i] = make_float2(0.5f * w.x, 0.5f * w.y);
  }
  float2 wreg[16];
  if constexpr (kWinRegs) {
#pragma unroll
    for (int n2 = 0; n2 < 16; ++n2) {
      const int c = tau + C::TPF * n2;
      const float2 w = *reinterpret_cast<const float2*>(p.window + 2 * c);
      wreg[n2] = make_float2(0.5f * w.x, 0.5f * w.y);
    }
  }
  Tw wtau;
  {
    float2 w;
    sincospif(-2.0f * (float)tau / (float)NFFT, &w.y, &w.x);
    wtau = make_tw<V>(w);
  }

  if (tid == 0) {
    mbar_init(&s_bar[0], 1);
    mbar_init(&s_bar[1], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  const int lead = p.lead;  // samples loaded ahead of the first frame (pre-emphasis history)
  const long n_tiles = p.n_tiles;

  // tile -> (clip, tile within clip), advanced by gridDim.x per iteration without dividing again
  long tile = blockIdx.x;
  const int tpc = p.tiles_per_clip;
  const int step_q = (int)(gridDim.x / (unsigned)tpc), step_r = (int)(gridDim.x % (unsigned)tpc);
  // variable-length batch: the last clip whose first tile is <= tl (clips without tiles are skipped over)
  auto locate = [&](long tl, int& c, int& t) {
    int lo = 0, hi = p.vl_clips - 1;
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if ((long)p.vl_first[mid] <= tl) lo = mid;
      else hi = mid - 1;
    }
    c = lo;
    t = (int)(tl - (long)p.vl_first[lo]);
  };
  int clip = (int)(tile / tpc), tin = (int)(tile % tpc);
  if (p.vl_first) locate(tile, clip, tin);
  auto next_tile = [&](int& c, int& t) {
    if (p.vl_first) {
      locate(tile + gridDim.x, c, t);
      return;
    }
    c += step_q;
    t += step_r;
    if (t >= tpc) {
      t -= tpc;
      ++c;
    }
  };
  // TF is a power of two
  int tf_shift = 0;
  while ((1 << tf_shift) < p.TF) ++tf_shift;
  if (p.use_tma && tid == 0 && tile < n_tiles) issue_span<NFFT>(&tmap, p, clip, tin << tf_shift, s_span, &s_bar[0]);

  int nclip = clip, ntin = tin;  // the tile after this one (prefetch target)
  for (int it = 0; tile < n_tiles; tile += gridDim.x, ++it, clip = nclip, tin = ntin) {
    const int b = p.span_bufs == 2 ? (it & 1) : 0;
    const int t0 = tin << tf_shift;
    nclip = clip;
    ntin = tin;
    next_tile(nclip, ntin);
    const long len = p.vl_len ? p.vl_len[clip] : p.n_samples;  // this clip's samples and frames
    const int Tc = p.vl_T ? p.vl_T[clip] : p.T;
    float* span = s_span + (size_t)b * p.span_alloc;
    // the span starts at the 16-byte aligned sample at or below the first needed one
    const int g_first = t0 * p.hop - NFFT / 2 - lead;
    const int shift = g_first - (g_first & ~3);
    float* ptile = s_ptile + (size_t)(p.pt_bufs == 2 ? (it & 1) : 0) * FP * p.ppitch;
    const TilePairs tpairs{ptile, p.ppitch, p.TF >> 1};
    const TileRows trows{ptile, p.ppitch};

    if (p.use_tma) {
      // two span buffers: prefetch the next tile into the other one now (its last readers
      // finished before the __syncthreads that closed the previous tile's FFT phase);
      // one span buffer: the prefetch is issued after this tile's FFT phase instead
      if (p.span_bufs == 2 && tid == 0 && tile + gridDim.x < n_tiles)
        issue_span<NFFT>(&tmap, p, nclip, ntin << tf_shift, s_span + (size_t)(b ^ 1) * p.span_alloc, &s_bar[b ^ 1]);
      mbar_wait(&s_bar[b], (uint32_t)(p.span_bufs == 2 ? (it >> 1) : it) & 1u);
      // variable-length batch: the TMA read the padded buffer, whose samples at and past the clip's end must read as
      // zero -- overwrite them before the frames load
      const long from = len - (long)(g_first & ~3);
      if (p.vl_len && from < p.span_alloc) {
        for (long i = max(0L, from) + tid; i < p.span_alloc; i += kThreads) span[i] = 0.0f;
        __syncthreads();
      }
    } else {
      // plain coalesced loader (clip stride or base not 16-byte aligned)
      const long g0 = (long)(g_first & ~3);
      const float* src = p.pcm + (size_t)clip * p.clip_stride;
      for (int i = tid; i < p.span_floats; i += kThreads) {
        const long n = g0 + i;
        span[i] = (n >= 0 && n < len) ? __ldg(src + n) : 0.0f;
      }
      __syncthreads();
    }

    // ---------------- FFT phase: FPI frames per iteration ----------------
    Xe* xb = s_xb + slot * C::XSTRIDE;
    auto fsync = [slot] { frame_sync<C::TPF>(slot); };
    for (int fi = 0; fi < ((p.debug_skip & 1) ? 0 : p.TF / FPI); ++fi) {
      const int f = (fi * SLOTS + slot) * TR::kFrames;  // first (or only) frame of this thread group
      const int off = shift + lead + f * p.hop;
      V v[16];
      if constexpr (!kWinRegs) {
#pragma unroll
        for (int n2 = 0; n2 < 16; ++n2) wreg[n2] = s_win[tau + C::TPF * n2];
      }
      if (p.preemph != 0.0f) {
        // samples from this frame's start to the end of the clip (frame start = f*hop - n_fft/2)
        const long n_valid = len - ((long)(t0 + f) * p.hop - NFFT / 2);
        ph_load_pre<NFFT>(v, span, off, p.hop, tau, wreg, p.preemph, n_valid);
      } else if (p.vec_ok && !(shift & 1)) {
        ph_load<NFFT, true>(v, span, off, p.hop, tau, wreg);
      } else {
        ph_load<NFFT, false>(v, span, off, p.hop, tau, wreg);
      }
      if (p.use_tma && p.span_bufs == 1 && p.early_tma && fi == p.TF / FPI - 1) {
        // every frame of the tile now sits in registers: the single span buffer is free, so the
        // next tile's PCM streams in underneath this tile's transform and mel projection
        __syncthreads();
        if (tid == 0 && tile + gridDim.x < n_tiles) issue_span<NFFT>(&tmap, p, nclip, ntin << tf_shift, s_span, &s_bar[0]);
      }
      ph_pass1<NFFT>(v, s_tw1, tau);
      if constexpr (TR::kXParts == 1) {
        fsync();  // previous iteration's readers of xb are done
        ph_x1_write<NFFT, 0>(v, xb, tau);
        fsync();
        ph_x1_read<NFFT, 0>(v, xb, tau);
      } else {
        fsync();
        ph_x1_write<NFFT, 1>(v, xb, tau);
        fsync();
        ph_x1_read<NFFT, 1>(v, xb, tau);
        fsync();
        ph_x1_write<NFFT, 2>(v, xb, tau);
        fsync();
        ph_x1_read<NFFT, 2>(v, xb, tau);
      }
      ph_pass2<NFFT>(v, s_tw2, tau);
      if constexpr (C::R3 > 1) {
        if constexpr (TR::kXParts == 1) {
          fsync();
          ph_x2_write<NFFT, 0>(v, xb, tau);
          fsync();
          ph_x2_read<NFFT, 0>(v, xb, tau);
        } else {
          fsync();
          ph_x2_write<NFFT, 1>(v, xb, tau);
          fsync();
          ph_x2_read<NFFT, 1>(v, xb, tau);
          fsync();
          ph_x2_write<NFFT, 2>(v, xb, tau);
          fsync();
          ph_x2_read<NFFT, 2>(v, xb, tau);
        }
        ph_pass3<NFFT>(v);
      }
      bool done = false;
      if constexpr (NFFT == 512) {
        if (p.split_regs) {
          // partner lane holds Z[M-k]: lane (16 - s) & 15 of the same half-warp, register 15 - r
          const int src = ((16 - tau) & 15) | (lane & 16);
          V bpart[8];
#pragma unroll
          for (int r = 0; r < 8; ++r) {
            const V sh = shfl_cx(v[15 - r], src);
            bpart[r] = (tau == 0) ? v[(16 - r) & 15] : sh;
          }
          if constexpr (MG)
            ph_split_regs512_to(v, bpart, tpairs, f, tau, wtau);
          else
            ph_split_regs512_to(v, bpart, trows, f, tau, wtau);
          done = true;
        }
      }
      if (!done) {
        V za[9], zb[8];
        if constexpr (TR::kXParts == 1) {
          fsync();
          ph_z_write<NFFT, 0>(v, xb, tau);
          fsync();
          ph_z_gather<NFFT, 0>(za, zb, xb, tau);
        } else {
          fsync();
          ph_z_write<NFFT, 1>(v, xb, tau);
          fsync();
          ph_z_gather<NFFT, 1>(za, zb, xb, tau);
          fsync();
          ph_z_write<NFFT, 2>(v, xb, tau);
          fsync();
          ph_z_gather<NFFT, 2>(za, zb, xb, tau);
        }
        if constexpr (MG)
          ph_split_pairs_to<NFFT>(za, zb, tpairs, f, tau, wtau);
        else
          ph_split_pairs_to<NFFT>(za, zb, trows, f, tau, wtau);
      }
    }
    __syncthreads();  // power tile complete
    if (p.use_tma && p.span_bufs == 1 && (!p.early_tma || (p.debug_skip & 1)) && tid == 0 && tile + gridDim.x < n_tiles)
      issue_span<NFFT>(&tmap, p, nclip, ntin << tf_shift, s_span, &s_bar[0]);  // (profiling mode without FFT phase)

    const int t_valid = min(p.TF, Tc - t0);
    if (p.power != nullptr) {
      float* dst = p.power + (size_t)clip * C::F * p.T + t0;
      for (int e = tid; e < C::F * p.TF; e += kThreads) {
        const int k = e / p.TF, t = e - k * p.TF;
        if (t < t_valid) dst[(size_t)k * p.T + t] = MG ? tpairs.get(k, t, TR::kFrames == 2) : trows.get(k, t);
      }
    }
    if constexpr (MG) {
      if (p.logmel != nullptr && !(p.debug_skip & 2)) {
        // ---------------- mel phase, grouped walk: lane -> tile column (one frame), worker -> band group
        const int c = lane & (p.TF - 1);
        const int half = p.TF >> 1;
        const int t = TR::kFrames == 2 ? ((c >= half ? c - half : c) << 1) + (c >= half ? 1 : 0) : c;  // frame of column c
        const int worker = (tid >> 5) * (32 >> tf_shift) + (lane >> tf_shift);
        const int m0 = s_mb[worker], m1 = s_mb[worker + 1];
        float mx = -FLT_MAX;
        if (m0 < m1 && t < t_valid) {
          float* dst = p.logmel + ((size_t)clip * p.n_mels + m0) * p.pitch + t0 + t;
          const float amin = p.amin;
          const int T = p.pitch;
          auto emit = [&](int, float val) {
            // 10*log10(x) = 10*log10(2) * log2(x); MUFU.LG2 is within 1e-6 dB here (x >= amin, never denormal)
            const float db = 3.01029995663981195f * fast_log2(fmaxf(amin, val));
            *dst = db;
            dst += T;
            mx = fmaxf(mx, db);
          };
          mel_groups(reinterpret_cast<const pk*>(ptile) + c, p.ppitch, s_mgseg, s_mgstep, reinterpret_cast<const pk2*>(s_mgw), m0,
                     m1, emit);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        if (lane == 0 && mx > -FLT_MAX) atomicMax(p.clipmax + clip, float_key(mx));
      }
    } else if (p.logmel != nullptr && p.mel_mma && !(p.debug_skip & 2)) {
      // ---------------- mel phase on the tensor cores.
      // D[frame][band] = P[frame][bin] * W[bin][band] in 16x8 output tiles.  Only the (n-tile,
      // k-tile) blocks of the filterbank that are not all zero are listed (n-major, built on the
      // host).  A unit = one 8-band n-tile x one 16-frame m-tile, owned by exactly one warp
      // (longest-processing-time assignment on the host), so the accumulators go from
      // registers through log10 straight to global memory: no atomics, no staging tile.
      const int warp = tid >> 5, g = lane >> 2, t4 = lane & 3;
      float mx = -FLT_MAX;
      for (int ui = 0; ui < kMaxUnits; ++ui) {
        const int unit = s_units[warp * kMaxUnits + ui];
        if (unit < 0) break;
        const int n = unit & 0xff, m = unit >> 8;
        // one accumulator per split term: three independent MMA chains instead of one
        float acc[4] = {0.0f, 0.0f, 0.0f, 0.0f}, acc_hl[4] = {0.0f, 0.0f, 0.0f, 0.0f},
              acc_lh[4] = {0.0f, 0.0f, 0.0f, 0.0f};
        const int q0 = s_npair[n], q1 = s_npair[n + 1];
        const float* pbase = ptile + t4 * p.ppitch + 16 * m + g;
        const int p4 = 4 * p.ppitch;
#pragma unroll 2
        for (int q = q0; q < q1; ++q) {
          const float2 bw = s_bw[q * 32 + lane];
          const float* pa = pbase + s_pk8[q] * 8 * p.ppitch;
          const float a[4] = {pa[0], pa[8], pa[p4], pa[p4 + 8]};
          uint32_t ah[4], al[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            ah[e] = __float_as_uint(a[e]) & 0xffffe000u;  // TF32 keeps 10 mantissa bits
            al[e] = __float_as_uint(a[e] - __uint_as_float(ah[e]));
          }
          const uint32_t bh0 = __float_as_uint(bw.x) & 0xffffe000u, bh1 = __float_as_uint(bw.y) & 0xffffe000u;
          const uint32_t bl0 = __float_as_uint(bw.x - __uint_as_float(bh0));
          const uint32_t bl1 = __float_as_uint(bw.y - __uint_as_float(bh1));
          mma_tf32(acc, ah, bh0, bh1);
          mma_tf32(acc_hl, ah, bl0, bl1);
          mma_tf32(acc_lh, al, bh0, bh1);
        }
        // acc: (frame g, band 2*t4), (g, 2*t4+1), (g+8, 2*t4), (g+8, 2*t4+1) of this unit
        const int tile = s_tile[n];
        const int band0 = (tile & 0xffff) + 2 * t4, nb = tile >> 16;
        float* orow = p.logmel + ((size_t)clip * p.n_mels + band0) * p.pitch + t0 + 16 * m + g;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int f = 16 * m + g + ((e & 2) ? 8 : 0);
          if (f < t_valid && 2 * t4 + (e & 1) < nb) {
            // 10*log10(x) = 10*log10(2) * log2(x); lg2.approx is within 1e-6 dB here (x >= amin, never denormal)
            const float val = acc[e] + (acc_hl[e] + acc_lh[e]);
            const float db = 3.01029995663981195f * fast_log2(fmaxf(p.amin, val));
            orow[((e & 1) ? p.pitch : 0) + ((e & 2) ? 8 : 0)] = db;
            mx = fmaxf(mx, db);
          }
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
      if (lane == 0 && mx > -FLT_MAX) atomicMax(p.clipmax + clip, float_key(mx));
    } else if (p.logmel != nullptr && !(p.debug_skip & 2)) {
      // ---------------- mel phase: lane -> frame, worker (warp or part of one) -> band group.
      // Band groups are balanced on the host by bins + bands (c_api.cu: band_split).
      const int t = lane & (p.TF - 1);
      const int worker = (tid >> 5) * (32 >> tf_shift) + (lane >> tf_shift);
      const int m0 = s_mb[worker], m1 = s_mb[worker + 1];
      float mx = -FLT_MAX;
      if (m0 < m1 && t < t_valid) {
        float* dst = p.logmel + ((size_t)clip * p.n_mels + m0) * p.pitch + t0 + t;
        const float amin = p.amin;
        const int T = p.pitch;
        auto emit = [&](int, float val) {
          // 10*log10(x) = 10*log10(2) * log2(x); MUFU.LG2 is within 1e-6 dB here (x >= amin, never denormal)
          const float db = 3.01029995663981195f * fast_log2(fmaxf(amin, val));
          *dst = db;
          dst += T;
          mx = fmaxf(mx, db);
        };
        if (p.ppitch == 34)  // 32-frame tiles
          mel_column<34>(ptile + t, 34, s_seg, s_w2, m0, m1, emit);
        else
          mel_column<0>(ptile + t, p.ppitch, s_seg, s_w2, m0, m1, emit);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
      if (lane == 0 && mx > -FLT_MAX) atomicMax(p.clipmax + clip, float_key(mx));
    }
    // with two power-tile buffers no barrier is needed here: the next tile writes
    // the other buffer and the tile after that is separated by the next tile's
    // __syncthreads; with one buffer the readers must drain first
    // One power-tile buffer: its readers must be done before the next tile's first split step
    // writes it.  A block barrier the next tile already has before that point does the job: the
    // one after the plain loader's fill, or the one after the span loads (single span buffer, early
    // prefetch) when the whole tile is transformed in one iteration; every other mode needs a
    // barrier of its own here.
    if (p.pt_bufs == 1 && p.use_tma && !(p.span_bufs == 1 && p.early_tma && p.TF == FPI)) __syncthreads();
  }
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------

size_t stft_mel_table_bytes(int n_fft, int n_mels, int mel_mma, int n_pairs, int n_tiles, int mel_groups, int mg_n) {
  const int F = n_fft / 2 + 1;
  if (mel_groups)
    return (size_t)mg_n * 32 + (size_t)(n_mels + 2) * 8 + (size_t)(n_mels + 3) * 8 + (size_t)(kMaxWorkers + 2) * 4;
  if (mel_mma)
    return (size_t)n_pairs * 32 * 8 + (size_t)n_pairs * 4 + (size_t)(2 * n_tiles + 1) * 4 + 8 * kMaxUnits * 4;
  return (size_t)F * 8 + (size_t)((n_mels + 2 + 1) & ~1) * 4 + (size_t)(kMaxWorkers + 2) * 4;
}

template <int NFFT>
static size_t smem_bytes_t(int span_alloc, int span_bufs, int ppitch, int pt_bufs, int packed, size_t mel_tab_bytes,
                           int threads, int mel_groups) {
  using C = FftCfg<NFFT>;
  const int SLOTS = threads / C::TPF;
  const int FP = mel_groups ? 4 * ((C::F + 3) / 4) : ((C::F + 7) & ~7);
  const size_t tw_bytes = packed ? sizeof(c2) : sizeof(float2);
  size_t b = 0;
  b += (size_t)span_bufs * span_alloc * 4;
  b += (size_t)((pt_bufs * FP * ppitch + 3) & ~3) * 4;
  b += (size_t)SLOTS * C::XSTRIDE * 8;
  b += (size_t)(C::TW1 + C::TW2) * tw_bytes;
  b += (size_t)C::M * 8;
  b += (mel_tab_bytes + 15) & ~(size_t)15;
  b += 16;
  return b;
}

template <int NFFT>
static void geometry_t(StftGeometry* g, int packed, int threads) {
  using C = FftCfg<NFFT>;
  g->tpf = C::TPF;
  g->fpi = (threads / C::TPF) * (packed ? 2 : 1);
  g->tw1 = C::TW1;
  g->tw2 = C::TW2;
  g->r3 = C::R3;
  g->m = C::M;
}

// two frames per thread group need <= 32 frames per iteration (one frame per lane in the mel phase)
bool stft_packed_supported(int n_fft) { return n_fft >= 512; }

int stft_geometry(int n_fft, int packed, int threads, StftGeometry* g) {
  switch (n_fft) {
    case 256: geometry_t<256>(g, packed, threads); return 0;
    case 512: geometry_t<512>(g, packed, threads); return 0;
    case 1024: geometry_t<1024>(g, packed, threads); return 0;
    case 2048: geometry_t<2048>(g, packed, threads); return 0;
    case 4096: geometry_t<4096>(g, packed, threads); return 0;
    default: return -1;
  }
}

size_t stft_smem_bytes(int n_fft, int span_alloc, int span_bufs, int ppitch, int pt_bufs, int packed,
                       size_t mel_tab_bytes, int threads, int mel_groups) {
  switch (n_fft) {
    case 256: return smem_bytes_t<256>(span_alloc, span_bufs, ppitch, pt_bufs, packed, mel_tab_bytes, threads, mel_groups);
    case 512: return smem_bytes_t<512>(span_alloc, span_bufs, ppitch, pt_bufs, packed, mel_tab_bytes, threads, mel_groups);
    case 1024: return smem_bytes_t<1024>(span_alloc, span_bufs, ppitch, pt_bufs, packed, mel_tab_bytes, threads, mel_groups);
    case 2048: return smem_bytes_t<2048>(span_alloc, span_bufs, ppitch, pt_bufs, packed, mel_tab_bytes, threads, mel_groups);
    case 4096: return smem_bytes_t<4096>(span_alloc, span_bufs, ppitch, pt_bufs, packed, mel_tab_bytes, threads, mel_groups);
    default: return 0;
  }
}

template <int NFFT, typename V, int THREADS, bool MG>
static cudaError_t launch_m(const CUtensorMap& tmap, const StftArgs& a, int grid, size_t smem, cudaStream_t st) {
  auto kfn = stft_mel_kernel<NFFT, V, THREADS, MG>;
  MMF_SMEM_ONCE(kfn, 227 * 1024);
  kfn<<<grid, THREADS, smem, st>>>(tmap, a);
  return cudaGetLastError();
}
template <int NFFT, typename V, int THREADS>
static cudaError_t launch_v(const CUtensorMap& tmap, const StftArgs& a, int grid, size_t smem, cudaStream_t st) {
  if (a.mel_groups) return launch_m<NFFT, V, THREADS, true>(tmap, a, grid, smem, st);
  return launch_m<NFFT, V, THREADS, false>(tmap, a, grid, smem, st);
}

template <int NFFT>
static cudaError_t launch_t(const CUtensorMap& tmap, const StftArgs& a, int grid, size_t smem, cudaStream_t st) {
  if constexpr (NFFT >= 1024) {  // 512-thread CTAs exist for the sizes that can need them
    if (a.threads == 512) {
      if (a.packed) return launch_v<NFFT, c2, 512>(tmap, a, grid, smem, st);
      return launch_v<NFFT, float2, 512>(tmap, a, grid, smem, st);
    }
  }
  if constexpr (NFFT >= 512) {
    if (a.packed) return launch_v<NFFT, c2, 256>(tmap, a, grid, smem, st);
  }
  return launch_v<NFFT, float2, 256>(tmap, a, grid, smem, st);
}

cudaError_t stft_mel_launch(int n_fft, const CUtensorMap& tmap, const StftArgs& a, int grid, size_t smem,
                            cudaStream_t st) {
  switch (n_fft) {
    case 256: return launch_t<256>(tmap, a, grid, smem, st);
    case 512: return launch_t<512>(tmap, a, grid, smem, st);
    case 1024: return launch_t<1024>(tmap, a, grid, smem, st);
    case 2048: return launch_t<2048>(tmap, a, grid, smem, st);
    case 4096: return launch_t<4096>(tmap, a, grid, smem, st);
    default: return cudaErrorInvalidValue;
  }
}

}  // namespace mmf
