// K3 and the generic kernels around the path: clamp + DCT-II (+ delta) in FP32 and on the
// tensor cores, the sequential zero-phase IIR (the chunk-parallel and fused forms live in
// change_fused.cu), derivative + norm, FIR filtfilt, stencils (get_velocity, Savitzky-Golay),
// the generic modulation-spectrum kernel (the fast ones live in modspec_fast.cu), RMS and
// Hilbert envelopes, find_peaks, PCM16 ingest and the polyphase resampler
// (script/mfcc.py:373-425, script/calc.py:221-343, :593-650; script/main.py:1566, :1601).
//
// These stages move ~0.3 MB per clip against 0.64 MB of PCM for the fused STFT
// kernel, so they are written for coalesced streaming access, not for math rate.
#include <cfloat>
#include <cstdint>
#include <cstring>

#include "fft_regs.cuh"
#include "mmf_internal.h"

namespace mmf {

__device__ __forceinline__ float key_to_float(int k) { return __int_as_float(k >= 0 ? k : k ^ 0x7FFFFFFF); }

// ---------------------------------------------------------------------------
// K3: top_db clamp + DCT-II (+ delta).  One thread per frame; the DCT rows sit in
// shared memory as [mel_chunk][NC] so each mel value feeds NC FMAs from broadcast
// 128-bit shared loads.  Block = 128 frames with a one-frame halo on each side
// when the delta (np.gradient) is requested.  T is the row pitch in frames; vT (a variable-length
// batch, else null) gives each clip's own frame count, 0 for a clip the launch skips.
// mel_chunk = n_mels unless the whole table does not fit shared memory (n_mfcc > 64 with n_mels >= 272):
// then the rows are staged mel_chunk at a time, and each coefficient still accumulates m = 0, 1, ... in order.
// ---------------------------------------------------------------------------
constexpr int kMfccThreads = 128;
constexpr size_t kMfccSmem = 200 * 1024;

template <int NC, bool VL>
__global__ void __launch_bounds__(kMfccThreads)
    mfcc_kernel(const float* __restrict__ dct_pad, int dct_pitch, float* logmel, const int* __restrict__ clipmax, long T,
                int n_mels, int n_mfcc, float top_db, float* __restrict__ mfcc, float* __restrict__ delta,
                int clamp_in_place, const int* __restrict__ vT, int mel_chunk) {
  extern __shared__ __align__(16) float sm[];
  float* s_dct = sm;                    // [mel_chunk][NC]
  float* s_col = sm + mel_chunk * NC;   // [NC][kMfccThreads + 1]
  const int tid = threadIdx.x;
  const long clip = blockIdx.y;
  const int halo = delta != nullptr ? 1 : 0;
  const int per_block = kMfccThreads - 2 * halo;
  const long Tn = VL ? vT[clip] : T;  // frames of this clip
  if (VL && (long)blockIdx.x * per_block >= Tn) return;

  const long t = (long)blockIdx.x * per_block - halo + tid;
  const bool valid = t >= 0 && t < Tn;
  const bool own = valid && tid >= halo && tid < kMfccThreads - halo;
  const float thr = top_db >= 0.0f ? key_to_float(clipmax[clip]) - top_db : -FLT_MAX;

  float acc[NC];
#pragma unroll
  for (int j = 0; j < NC; ++j) acc[j] = 0.0f;
  float* col = logmel + (size_t)clip * n_mels * T + (valid ? t : 0);
  // every thread of the block takes every chunk's barriers; only frames of the clip read and accumulate
  for (int c0 = 0; c0 < n_mels; c0 += mel_chunk) {
    const int c1 = min(n_mels, c0 + mel_chunk);
    if (c0 > 0) __syncthreads();  // the previous chunk's rows have been read by every thread
    for (int i = tid; i < (c1 - c0) * NC; i += kMfccThreads) {
      const int m = i / NC, j = i - m * NC;
      s_dct[i] = dct_pad[(c0 + m) * dct_pitch + j];
    }
    __syncthreads();
    if (!valid) continue;
    // software pipeline: the next 8 mel rows are in flight while the current 8 feed their FMAs
    // (the kernel is a pure stream: 4*n_mels bytes in, 8*n_mfcc bytes out per frame)
    float cur[8], nxt[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) cur[u] = (c0 + u < c1) ? __ldcs(col + (size_t)(c0 + u) * T) : 0.0f;
    for (int m0 = c0; m0 < c1; m0 += 8) {
#pragma unroll
      for (int u = 0; u < 8; ++u) nxt[u] = (m0 + 8 + u < c1) ? __ldcs(col + (size_t)(m0 + 8 + u) * T) : 0.0f;
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int m = m0 + u;
        if (m < c1) {
          const float x = fmaxf(cur[u], thr);
          if (clamp_in_place && own) col[(size_t)m * T] = x;
          const float4* d4 = reinterpret_cast<const float4*>(s_dct + (m - c0) * NC);
#pragma unroll
          for (int j4 = 0; j4 < NC / 4; ++j4) {
            const float4 d = d4[j4];
            acc[4 * j4 + 0] = fmaf(d.x, x, acc[4 * j4 + 0]);
            acc[4 * j4 + 1] = fmaf(d.y, x, acc[4 * j4 + 1]);
            acc[4 * j4 + 2] = fmaf(d.z, x, acc[4 * j4 + 2]);
            acc[4 * j4 + 3] = fmaf(d.w, x, acc[4 * j4 + 3]);
          }
        }
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) cur[u] = nxt[u];
    }
  }
  if (own) {
    float* dst = mfcc + (size_t)clip * n_mfcc * T + t;
#pragma unroll
    for (int j = 0; j < NC; ++j)
      if (j < n_mfcc) dst[(size_t)j * T] = acc[j];
  }
  if (delta != nullptr) {
#pragma unroll
    for (int j = 0; j < NC; ++j) s_col[j * (kMfccThreads + 1) + tid] = acc[j];
    __syncthreads();
    if (own) {
      float* dst = delta + (size_t)clip * n_mfcc * T + t;
#pragma unroll
      for (int j = 0; j < NC; ++j) {
        if (j < n_mfcc) {
          const float* c = s_col + j * (kMfccThreads + 1) + tid;
          float d;
          if (Tn == 1) {
            d = 0.0f;
          } else if (t == 0) {
            d = c[1] - c[0];
          } else if (t == Tn - 1) {
            d = c[0] - c[-1];
          } else {
            d = (c[1] - c[-1]) / 2.0f;
          }
          dst[(size_t)j * T] = d;
        }
      }
    }
  }
}

// K3, fast form for n_mfcc <= 32 and n_mels a multiple of 8 (every BASELINE shape; PITCH = padded table row: 16 or 32
// coefficients): same thread-per-frame layout and
// the same FMA order as mfcc_kernel (so the MFCCs are bit-identical), but coefficient PAIRS are accumulated with
// packed FFMA2 (half the issue slots of the contraction), the mel rows are walked with pointer steps instead of
// 64-bit index products, and the loop body carries no predicates.  ncu of mfcc_kernel<16> on the bench shape:
// 83.4 M warp instructions of which 21 M are the FFMAs -- issue-bound at 95 us for a 271 MB stream.
template <int NP, int PITCH, bool VL>
__global__ void __launch_bounds__(kMfccThreads)
    mfcc_pk_kernel(const float* __restrict__ dct_pad, float* logmel, const int* __restrict__ clipmax, long T, int n_mels,
                   int n_mfcc, float top_db, float* __restrict__ mfcc, float* __restrict__ delta, int clamp_in_place,
                   const int* __restrict__ vT) {
  extern __shared__ __align__(16) float sm[];
  static_assert(2 * NP <= PITCH, "coefficient pairs must fit the padded table row");
  float* s_dct = sm;                    // [n_mels][PITCH]
  float* s_col = sm + n_mels * PITCH;   // [2 NP][kMfccThreads + 1]
  const int tid = threadIdx.x;
  const long clip = blockIdx.y;
  const int halo = delta != nullptr ? 1 : 0;
  const int per_block = kMfccThreads - 2 * halo;
  const long Tn = VL ? vT[clip] : T;  // frames of this clip
  if (VL && (long)blockIdx.x * per_block >= Tn) return;
  for (int i = tid; i < n_mels * (PITCH / 4); i += kMfccThreads)
    reinterpret_cast<float4*>(s_dct)[i] = reinterpret_cast<const float4*>(dct_pad)[i];
  __syncthreads();

  const int Ti = (int)T;  // row pitch as a 32-bit value: u * Ti is one IMAD.WIDE per address instead of a 64-bit product
  const long t = (long)blockIdx.x * per_block - halo + tid;
  const bool valid = t >= 0 && t < Tn;
  const bool own = valid && tid >= halo && tid < kMfccThreads - halo;
  const float thr = top_db >= 0.0f ? key_to_float(clipmax[clip]) - top_db : -FLT_MAX;

  pk acc[NP];
#pragma unroll
  for (int j = 0; j < NP; ++j) acc[j] = pmake(0.0f, 0.0f);
  // frames outside the clip (halo of the first / last block) read frame 0 / T - 1: finite, never stored
  const long tc = t < 0 ? 0 : (t >= Tn ? Tn - 1 : t);
  float* col = logmel + (size_t)clip * n_mels * T + tc;
  const bool store_clamped = clamp_in_place && own;
  {
    const int T8 = 8 * Ti;
    float cur[8], nxt[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) cur[u] = __ldcs(col + u * Ti);
    const float* s_row = s_dct;
    for (int m0 = 0; m0 < n_mels; m0 += 8) {
      float* nrow = col + T8;
      if (m0 + 8 < n_mels) {
#pragma unroll
        for (int u = 0; u < 8; ++u) nxt[u] = __ldcs(nrow + u * Ti);
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const float x = fmaxf(cur[u], thr);
        if (store_clamped) col[u * Ti] = x;
        const pk xx = pmake(x, x);
        const float4* d4 = reinterpret_cast<const float4*>(s_row + PITCH * u);
#pragma unroll
        for (int j4 = 0; j4 < (NP + 1) / 2; ++j4) {
          const float4 d = d4[j4];
          acc[2 * j4] = sfma(pmake(d.x, d.y), xx, acc[2 * j4]);
          if (2 * j4 + 1 < NP) acc[2 * j4 + 1] = sfma(pmake(d.z, d.w), xx, acc[2 * j4 + 1]);
        }
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) cur[u] = nxt[u];
      col = nrow;
      s_row += 8 * PITCH;
    }
  }
  float out[2 * NP];
#pragma unroll
  for (int j = 0; j < NP; ++j) {
    out[2 * j] = plo(acc[j]);
    out[2 * j + 1] = phi(acc[j]);
  }
  if (own) {
    float* dst = mfcc + (size_t)clip * n_mfcc * T + t;
#pragma unroll
    for (int j = 0; j < 2 * NP; ++j) {
      if (j < n_mfcc) *dst = out[j];
      dst += Ti;
    }
  }
  if (delta != nullptr) {
#pragma unroll
    for (int j = 0; j < 2 * NP; ++j) s_col[j * (kMfccThreads + 1) + tid] = out[j];
    __syncthreads();
    if (own) {
      float* dst = delta + (size_t)clip * n_mfcc * T + t;
      // np.gradient: one-sided at the clip's ends, central inside
      const int lo = t == 0 ? 0 : -1, hi = t == Tn - 1 ? 0 : 1;
      const float scale = (lo != 0 && hi != 0) ? 0.5f : 1.0f;
#pragma unroll
      for (int j = 0; j < 2 * NP; ++j) {
        if (j < n_mfcc) {
          const float* c = s_col + j * (kMfccThreads + 1) + tid;
          // (c[1] - c[-1]) / 2 and (c[1] - c[0]) / 1 exactly as mfcc_kernel: division by 2 = multiplication by 0.5
          *dst = Tn == 1 ? 0.0f : (c[hi] - c[lo]) * scale;
        }
        dst += Ti;
      }
    }
  }
}

cudaError_t mfcc_launch(const float* dct_pad, int nc_pad, float* logmel, const int* clipmax, long n_clips, long T,
                        int n_mels, int n_mfcc, float top_db, float* mfcc, float* delta, int clamp_in_place,
                        cudaStream_t st, const int* vT) {
  const int halo = delta != nullptr ? 1 : 0;
  const int per_block = kMfccThreads - 2 * halo;
  dim3 grid((unsigned)((T + per_block - 1) / per_block), (unsigned)n_clips);
  int nc = n_mfcc <= 16 ? 16 : (n_mfcc <= 32 ? 32 : (n_mfcc <= 64 ? 64 : 128));
  // DCT rows that fit beside the delta tile: every n_mels up to 512 for nc <= 64, 271 for nc = 128
  const int mel_chunk = std::min<int>(n_mels, (int)(kMfccSmem / sizeof(float) / nc) - (kMfccThreads + 1));
  size_t smem = ((size_t)mel_chunk * nc + (size_t)nc * (kMfccThreads + 1)) * sizeof(float);
  if ((nc == 16 || nc == 32) && nc_pad == nc && n_mels % 8 == 0 && n_mels >= 8 && T < (1L << 27)) {
    const int np = n_mfcc <= 8 ? 4 : (n_mfcc + 1) / 2;
#define MMF_MFCC_PK_LAUNCH(N, P, V)                                                                                \
  {                                                                                                                \
    auto kfn = mfcc_pk_kernel<N, P, V>;                                                                            \
    MMF_SMEM_ONCE(kfn, 200 * 1024);                                                                                \
    kfn<<<grid, kMfccThreads, smem, st>>>(dct_pad, logmel, clipmax, T, n_mels, n_mfcc, top_db, mfcc, delta,        \
                                          clamp_in_place, vT);                                                     \
  }
#define MMF_MFCC_PK_CASE(N, P)                                                                                     \
  case N: {                                                                                                        \
    if (vT) MMF_MFCC_PK_LAUNCH(N, P, true)                                                                         \
    else MMF_MFCC_PK_LAUNCH(N, P, false)                                                                           \
    break;                                                                                                         \
  }
    switch (np) {
      MMF_MFCC_PK_CASE(4, 16)
      MMF_MFCC_PK_CASE(5, 16)
      MMF_MFCC_PK_CASE(6, 16)
      MMF_MFCC_PK_CASE(7, 16)
      MMF_MFCC_PK_CASE(8, 16)
      MMF_MFCC_PK_CASE(9, 32)
      MMF_MFCC_PK_CASE(10, 32)
      MMF_MFCC_PK_CASE(11, 32)
      MMF_MFCC_PK_CASE(12, 32)
      MMF_MFCC_PK_CASE(13, 32)
      MMF_MFCC_PK_CASE(14, 32)
      MMF_MFCC_PK_CASE(15, 32)
      MMF_MFCC_PK_CASE(16, 32)
    }
#undef MMF_MFCC_PK_CASE
#undef MMF_MFCC_PK_LAUNCH
    count_launch();
    return cudaGetLastError();
  }
#define MMF_MFCC_LAUNCH(N, V)                                                                                    \
  {                                                                                                              \
    auto kfn = mfcc_kernel<N, V>;                                                                                \
    MMF_SMEM_ONCE(kfn, kMfccSmem);                                                                               \
    kfn<<<grid, kMfccThreads, smem, st>>>(dct_pad, nc_pad, logmel, clipmax, T, n_mels, n_mfcc, top_db, mfcc,     \
                                          delta, clamp_in_place, vT, mel_chunk);                                 \
  }
#define MMF_MFCC_CASE(N)                                                                                         \
  case N: {                                                                                                      \
    if (vT) MMF_MFCC_LAUNCH(N, true)                                                                             \
    else MMF_MFCC_LAUNCH(N, false)                                                                               \
    break;                                                                                                       \
  }
  switch (nc) {
    MMF_MFCC_CASE(16)
    MMF_MFCC_CASE(32)
    MMF_MFCC_CASE(64)
    MMF_MFCC_CASE(128)
  }
#undef MMF_MFCC_CASE
#undef MMF_MFCC_LAUNCH
  count_launch();
  return cudaGetLastError();
}

// Variable-length batch: every output element at or past its clip's frame count is 0.  One CTA per clip; the
// kernels before it write frames [0, T[clip]) only.
__global__ void varlen_tails_kernel(const int* __restrict__ T, int pitch, double* __restrict__ tot,
                                    float* __restrict__ logmel, int n_mels, float* __restrict__ mfcc,
                                    float* __restrict__ delta, int n_mfcc) {
  const long clip = blockIdx.x;
  const int t0 = T[clip], w = pitch - t0;
  if (w <= 0) return;
  for (int i = threadIdx.x; i < w; i += blockDim.x) tot[(size_t)clip * pitch + t0 + i] = 0.0;
  auto zero = [&](float* buf, int rows) {  // rows x w can pass 2^31 (long clips at small hops): 64-bit indices
    if (!buf) return;
    for (long e = threadIdx.x; e < (long)rows * w; e += blockDim.x) {
      const long r = e / w;
      buf[((size_t)clip * rows + r) * pitch + t0 + (e - r * w)] = 0.0f;
    }
  };
  zero(logmel, n_mels);
  zero(mfcc, n_mfcc);
  zero(delta, n_mfcc);
}

cudaError_t varlen_tails_launch(long n_clips, const int* T, int pitch, double* tot, float* logmel, int n_mels,
                                float* mfcc, float* delta, int n_mfcc, cudaStream_t st) {
  varlen_tails_kernel<<<(unsigned)n_clips, 256, 0, st>>>(T, pitch, tot, logmel, n_mels, mfcc, delta, n_mfcc);
  count_launch();
  return cudaGetLastError();
}

// Variable-length K6 batch: windows [n_win[clip], W) of every magnitude row [n_coef][W][nb] and of the band rows
// [W][n_bands] are 0.  One CTA per clip; the kernels before it write windows [0, n_win[clip]) only.
__global__ void modspec_tails_kernel(const int* __restrict__ n_win, long W, float* __restrict__ mag, int n_coef, int nb,
                                     float* __restrict__ band, int n_bands) {
  const long clip = blockIdx.x;
  const long w0 = n_win[clip];
  if (w0 >= W) return;
  if (mag) {
    const long row = (W - w0) * nb;  // tail floats of one coefficient's row
    for (long e = threadIdx.x; e < (long)n_coef * row; e += blockDim.x) {
      const long c = e / row;
      mag[(((size_t)clip * n_coef + c) * W + w0) * nb + (e - c * row)] = 0.0f;
    }
  }
  if (band)
    for (long e = threadIdx.x; e < (W - w0) * n_bands; e += blockDim.x) band[((size_t)clip * W + w0) * n_bands + e] = 0.0f;
}

cudaError_t modspec_tails_launch(long n_clips, const int* n_win, long W, float* mag, int n_coef, int nb, float* band,
                                 int n_bands, cudaStream_t st) {
  modspec_tails_kernel<<<(unsigned)n_clips, 256, 0, st>>>(n_win, W, mag, n_coef, nb, band, n_bands);
  count_launch();
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// K3 on the tensor cores: [frames x n_mels] . [n_mels x n_mfcc] with mma.sync m16n8k8 TF32 and
// the 3-term operand split (hi*hi + hi*lo + lo*hi into independent fp32 accumulators, ~2^-21
// relative per product; single-pass TF32 misses the 1e-3 MFCC tolerance by 27x, SURVEY 7.4-1).
// The FP32 kernel above is bound by instruction issue (83 % of the issue slots, 640 FFMAs per
// frame); here the contraction is 60 MMAs per 32 frames and the kernel goes back to being a stream.
//   A (m16 x k8) = clamped log-mel, rows = frames, straight from global memory (each element is
//                  needed by exactly one lane; 8 consecutive frames per mel row = one 32-byte sector),
//   B (k8 x n8)  = DCT-II rows, pre-split hi/lo in fragment order in shared memory,
//   D (m16 x n8) -> a per-warp [NC][34] tile in shared memory, from which MFCC and its np.gradient
//                  delta leave as coalesced 128-byte rows (one frame of halo on each side).
// One warp = 32 frames (30 owned + halo) of one clip.
// ---------------------------------------------------------------------------
constexpr int kMmaWarps = 4;
constexpr int kMmaOwn = 30;  // frames owned per warp when the delta is requested (else 32)

__device__ __forceinline__ void mma_tf32_16x8x8(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, "
      "{%0, %1, %2, %3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// NT = n-tiles of 8 coefficients (n_mfcc <= 8*NT)
template <int NT>
__global__ void __launch_bounds__(kMmaWarps * 32)
    mfcc_mma_kernel(const float4* __restrict__ bfrag, float* logmel, const int* __restrict__ clipmax, long T, int n_mels,
                    int n_mfcc, float top_db, float* __restrict__ mfcc, float* __restrict__ delta, int clamp_in_place) {
  extern __shared__ __align__(16) float sm_mma[];
  const int ksteps = (n_mels + 7) / 8;
  float4* s_b = reinterpret_cast<float4*>(sm_mma);                 // [ksteps][NT][32] (hi0, hi1, lo0, lo1)
  float* s_c = sm_mma + (size_t)ksteps * NT * 32 * 4;              // [kMmaWarps][8*NT][34]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t4 = lane & 3;
  for (int i = tid; i < ksteps * NT * 32; i += kMmaWarps * 32) s_b[i] = bfrag[i];
  __syncthreads();
  const long clip = blockIdx.y;
  const int halo = delta != nullptr ? 1 : 0;
  const int own = delta != nullptr ? kMmaOwn : 32;
  const long t_base = ((long)blockIdx.x * kMmaWarps + warp) * own - halo;  // first frame of this warp's 32
  if (t_base >= T) return;
  const float thr = top_db >= 0.0f ? key_to_float(clipmax[clip]) - top_db : -FLT_MAX;
  float* lm = logmel + (size_t)clip * n_mels * T;
  float acc[2][NT][3][4];
#pragma unroll
  for (int m = 0; m < 2; ++m)
#pragma unroll
    for (int n = 0; n < NT; ++n)
#pragma unroll
      for (int q = 0; q < 3; ++q)
#pragma unroll
        for (int e = 0; e < 4; ++e) acc[m][n][q][e] = 0.0f;
  // frames of this lane's fragment rows: t_base + 16*m + g (+8)
  for (int ks = 0; ks < ksteps; ++ks) {
    uint32_t ah[2][4], al[2][4];
#pragma unroll
    for (int m = 0; m < 2; ++m)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const long t = t_base + 16 * m + g + ((e & 1) ? 8 : 0);
        const int mel = 8 * ks + t4 + ((e & 2) ? 4 : 0);
        float x = 0.0f;
        if (t >= 0 && t < T && mel < n_mels) {
          float* src = lm + (size_t)mel * T + t;
          x = fmaxf(__ldcs(src), thr);
          // the clamp is written back by the lanes that own the frame (halo frames belong to a neighbour)
          if (clamp_in_place && t >= t_base + halo && t < t_base + halo + own) *src = x;
        }
        ah[m][e] = __float_as_uint(x) & 0xffffe000u;
        al[m][e] = __float_as_uint(x - __uint_as_float(ah[m][e]));
      }
#pragma unroll
    for (int n = 0; n < NT; ++n) {
      const float4 b = s_b[(ks * NT + n) * 32 + lane];
      const uint32_t bh0 = __float_as_uint(b.x), bh1 = __float_as_uint(b.y);
      const uint32_t bl0 = __float_as_uint(b.z), bl1 = __float_as_uint(b.w);
#pragma unroll
      for (int m = 0; m < 2; ++m) {
        mma_tf32_16x8x8(acc[m][n][0], ah[m], bh0, bh1);
        mma_tf32_16x8x8(acc[m][n][1], ah[m], bl0, bl1);
        mma_tf32_16x8x8(acc[m][n][2], al[m], bh0, bh1);
      }
    }
  }
  // D fragments -> s_c[coef][local frame]: (frame g, coef 2*t4), (g, 2*t4+1), (g+8, 2*t4), (g+8, 2*t4+1)
  float* c = s_c + (size_t)warp * (8 * NT) * 34;
#pragma unroll
  for (int m = 0; m < 2; ++m)
#pragma unroll
    for (int n = 0; n < NT; ++n)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float v = acc[m][n][0][e] + (acc[m][n][1][e] + acc[m][n][2][e]);
        c[(8 * n + 2 * t4 + (e & 1)) * 34 + 16 * m + g + ((e & 2) ? 8 : 0)] = v;
      }
  __syncwarp();
  // lane = local frame; owned frames leave as coalesced rows
  const long t = t_base + lane;
  const bool mine = lane >= halo && lane < halo + own && t < T;
  if (mine) {
    for (int j = 0; j < n_mfcc; ++j) {
      const float* cj = c + j * 34 + lane;
      mfcc[((size_t)clip * n_mfcc + j) * T + t] = cj[0];
      if (delta != nullptr) {
        float d;
        if (T == 1) {
          d = 0.0f;
        } else if (t == 0) {
          d = cj[1] - cj[0];
        } else if (t == T - 1) {
          d = cj[0] - cj[-1];
        } else {
          d = (cj[1] - cj[-1]) / 2.0f;
        }
        delta[((size_t)clip * n_mfcc + j) * T + t] = d;
      }
    }
  }
}

// B fragments of the DCT for the MMA kernel: [ksteps][NT][32 lanes] (hi0, hi1, lo0, lo1);
// b0 = D[coef 8n + lane/4][mel 8ks + lane%4], b1 = ... mel + 4
void mfcc_mma_bfrag(const float* dct /* [n_mfcc][n_mels] */, int n_mfcc, int n_mels, std::vector<float4>& out) {
  const int ksteps = (n_mels + 7) / 8, NT = (n_mfcc + 7) / 8;
  out.assign((size_t)ksteps * NT * 32, make_float4(0.f, 0.f, 0.f, 0.f));
  auto at = [&](int coef, int mel) { return (coef < n_mfcc && mel < n_mels) ? dct[(size_t)coef * n_mels + mel] : 0.0f; };
  auto hi = [](float w) {
    uint32_t u;
    memcpy(&u, &w, 4);
    u &= 0xffffe000u;
    float h;
    memcpy(&h, &u, 4);
    return h;
  };
  for (int ks = 0; ks < ksteps; ++ks)
    for (int n = 0; n < NT; ++n)
      for (int lane = 0; lane < 32; ++lane) {
        const int g = lane >> 2, t4 = lane & 3;
        const float w0 = at(8 * n + g, 8 * ks + t4), w1 = at(8 * n + g, 8 * ks + t4 + 4);
        const float h0 = hi(w0), h1 = hi(w1);
        out[((size_t)ks * NT + n) * 32 + lane] = make_float4(h0, h1, w0 - h0, w1 - h1);
      }
}

bool mfcc_mma_supported(int n_mfcc, int n_mels) { return n_mfcc <= 32 && n_mels <= 512; }

cudaError_t mfcc_mma_launch(const float4* bfrag_dev, float* logmel, const int* clipmax, long n_clips, long T, int n_mels,
                            int n_mfcc, float top_db, float* mfcc, float* delta, int clamp_in_place, cudaStream_t st) {
  const int NT = (n_mfcc + 7) / 8, ksteps = (n_mels + 7) / 8;
  const int own = delta != nullptr ? kMmaOwn : 32;
  const long per_block = (long)kMmaWarps * own;
  dim3 grid((unsigned)((T + (delta != nullptr ? 1 : 0) + per_block - 1) / per_block), (unsigned)n_clips);
  const size_t smem = (size_t)ksteps * NT * 32 * 16 + (size_t)kMmaWarps * 8 * NT * 34 * 4;
#define MMF_MMA_CASE(N)                                                                                          \
  case N: {                                                                                                      \
    MMF_SMEM_ONCE(mfcc_mma_kernel<N>, 200 * 1024);                                                               \
    mfcc_mma_kernel<N><<<grid, kMmaWarps * 32, smem, st>>>(bfrag_dev, logmel, clipmax, T, n_mels, n_mfcc, top_db, \
                                                         mfcc, delta, clamp_in_place);                           \
    break;                                                                                                       \
  }
  switch (NT) {
    MMF_MMA_CASE(1)
    MMF_MMA_CASE(2)
    MMF_MMA_CASE(3)
    MMF_MMA_CASE(4)
    default: return cudaErrorInvalidValue;
  }
#undef MMF_MMA_CASE
  count_launch();
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// K4: scipy.signal.sosfiltfilt along time, float64 (script/mfcc.py:402, :421).
// Odd extension (padlen samples each side, computed in the input dtype as scipy
// does), zi * first sample, forward cascade, same backwards, trim.
//
// One warp owns 32 rows.  The recurrence is sequential in time, so each lane walks
// its own row -- but rows are time-major in memory, so the warp stages
// [32 rows x 32 samples] tiles through shared memory: global loads and stores are
// coalesced 128/256-byte row segments and the per-sample loop only touches shared
// memory.  The forward result of the T interior samples is parked in y and
// overwritten in place by the backward pass; the forward output over the right
// extension (needed to start the backward pass) stays in shared memory.
// ---------------------------------------------------------------------------
constexpr int kSosChunk = 32;

template <typename TIn, int NS>
__global__ void __launch_bounds__(32)
    sosfiltfilt_kernel(const TIn* __restrict__ x, long rows, long T, long x_row_stride, int group_rows,
                       long group_stride, const SosArgs a, double* __restrict__ y, long y_row_stride) {
  extern __shared__ __align__(16) double sm_d[];
  constexpr int CH = kSosChunk;
  const int p = a.padlen;
  double* tile = sm_d;                    // [32][CH + 1]
  double* tail = sm_d + 32 * (CH + 1);    // [32][p + 1]
  long* s_off = reinterpret_cast<long*>(tail + 32 * (p + 1));  // [32] element offset of each row in x
  const int lane = threadIdx.x;
  const long row0 = (long)blockIdx.x * 32;
  const int nrows = (int)min(32L, rows - row0);
  const int ns = NS > 0 ? NS : a.n_sections;
  constexpr int ZS = NS > 0 ? NS : 16;
  double z0[ZS], z1[ZS];

  {
    const long rr = row0 + (lane < nrows ? lane : 0);
    const long g = rr / group_rows, gi = rr - g * group_rows;
    s_off[lane] = g * group_stride + gi * x_row_stride;
  }
  __syncwarp();
  auto row_ptr = [&](int r) -> const TIn* { return x + s_off[r]; };
  auto cascade = [&](double v) -> double {
#pragma unroll
    for (int s = 0; s < ZS; ++s) {
      if (s < ns) {
        const double out = fma(a.sos[s][0], v, z0[s]);
        z0[s] = fma(a.sos[s][1], v, fma(-a.sos[s][4], out, z1[s]));
        z1[s] = fma(a.sos[s][2], v, -a.sos[s][5] * out);
        v = out;
      }
    }
    return v;
  };

  const bool mine = lane < nrows;
  const TIn* xme = row_ptr(mine ? lane : 0);
  const TIn x0 = xme[0], xl = xme[T - 1];
  const TIn two = (TIn)2;
  const long L = T + 2L * p;

  // Row r's sample for extended index i (odd extension computed in the input dtype).
  // All 32 row loads of a chunk are issued back to back (32 independent requests in
  // flight per lane) and the next chunk is fetched while the current one is filtered.
  const TIn rx0_all = x0, rxl_all = xl;
  auto fetch_fwd = [&](long c0, TIn (&vals)[32]) {
    const long i = c0 + lane;
#pragma unroll
    for (int r = 0; r < 32; ++r) {
      const TIn rx0 = __shfl_sync(0xffffffffu, rx0_all, r), rxl = __shfl_sync(0xffffffffu, rxl_all, r);
      TIn v = (TIn)0;
      if (r < nrows && i < L) {
        const TIn* xr = x + s_off[r];
        if (i < p) {
          v = (TIn)(two * rx0 - xr[p - i]);
        } else if (i < p + T) {
          v = xr[i - p];
        } else {
          v = (TIn)(two * rxl - xr[T - 2 - (i - p - T)]);
        }
      }
      vals[r] = v;
    }
  };

  // ---- forward pass over [left ext | x | right ext]
  {
    const double e0 = (double)(TIn)(two * x0 - xme[p]);
#pragma unroll
    for (int s = 0; s < ZS; ++s)
      if (s < ns) {
        z0[s] = a.zi[s][0] * e0;
        z1[s] = a.zi[s][1] * e0;
      }
  }
  {
    TIn cur[32], nxt[32];
    fetch_fwd(0, cur);
    for (long c0 = 0; c0 < L; c0 += CH) {
      const long i = c0 + lane;
#pragma unroll
      for (int r = 0; r < 32; ++r) tile[r * (CH + 1) + lane] = (double)cur[r];
      if (c0 + CH < L) fetch_fwd(c0 + CH, nxt);
      __syncwarp();
      if (mine) {
        const int n = (int)min((long)CH, L - c0);
        double* trow = tile + lane * (CH + 1);
#pragma unroll 4
        for (int k = 0; k < n; ++k) trow[k] = cascade(trow[k]);
      }
      __syncwarp();
      if (i >= p && i < p + T) {
#pragma unroll
        for (int r = 0; r < 32; ++r)
          if (r < nrows) y[(row0 + r) * y_row_stride + (i - p)] = tile[r * (CH + 1) + lane];
      } else if (i >= p + T && i < L) {
#pragma unroll
        for (int r = 0; r < 32; ++r)
          if (r < nrows) tail[r * (p + 1) + (int)(i - p - T)] = tile[r * (CH + 1) + lane];
      }
      __syncwarp();
#pragma unroll
      for (int r = 0; r < 32; ++r) cur[r] = nxt[r];
    }
  }

  // ---- backward pass, from the end of the right extension down to the first interior sample
  {
    const double f0 = tail[(mine ? lane : 0) * (p + 1) + p - 1];
#pragma unroll
    for (int s = 0; s < ZS; ++s)
      if (s < ns) {
        z0[s] = a.zi[s][0] * f0;
        z1[s] = a.zi[s][1] * f0;
      }
  }
  auto fetch_bwd = [&](long c0, double (&vals)[32]) {
    const long i = c0 - lane;
#pragma unroll
    for (int r = 0; r < 32; ++r) {
      double v = 0.0;
      if (r < nrows && i >= p)
        v = i >= p + T ? tail[r * (p + 1) + (int)(i - p - T)] : y[(row0 + r) * y_row_stride + (i - p)];
      vals[r] = v;
    }
  };
  {
    double cur[32], nxt[32];
    fetch_bwd(L - 1, cur);
    for (long c0 = L - 1; c0 >= p; c0 -= CH) {
      const long i = c0 - lane;
#pragma unroll
      for (int r = 0; r < 32; ++r) tile[r * (CH + 1) + lane] = cur[r];
      if (c0 - CH >= p) fetch_bwd(c0 - CH, nxt);
      __syncwarp();
      if (mine) {
        const int n = (int)min((long)CH, c0 - p + 1);
        double* trow = tile + lane * (CH + 1);
#pragma unroll 4
        for (int k = 0; k < n; ++k) trow[k] = cascade(trow[k]);
      }
      __syncwarp();
      if (i >= p && i < p + T) {
#pragma unroll
        for (int r = 0; r < 32; ++r)
          if (r < nrows) y[(row0 + r) * y_row_stride + (i - p)] = tile[r * (CH + 1) + lane];
      }
      __syncwarp();
#pragma unroll
      for (int r = 0; r < 32; ++r) cur[r] = nxt[r];
    }
  }
}

template <typename TIn>
static cudaError_t sos_launch_t(const TIn* x, long rows, long T, long xs, int group_rows, long group_stride,
                                const SosArgs& a, double* y, long ys, cudaStream_t st) {
  const int threads = 32;
  const unsigned grid = (unsigned)((rows + 31) / 32);
  const size_t smem = (size_t)(32 * (kSosChunk + 1) + 32 * (a.padlen + 1) + 32) * sizeof(double);
  switch (a.n_sections) {
#define MMF_SOS_CASE(N)                                                                                             \
  case N:                                                                                                           \
    sosfiltfilt_kernel<TIn, N><<<grid, threads, smem, st>>>(x, rows, T, xs, group_rows, group_stride, a, y, ys);    \
    break;
    MMF_SOS_CASE(1)
    MMF_SOS_CASE(2)
    MMF_SOS_CASE(3)
    MMF_SOS_CASE(4)
    MMF_SOS_CASE(5)
    MMF_SOS_CASE(6)
    MMF_SOS_CASE(7)
    MMF_SOS_CASE(8)
#undef MMF_SOS_CASE
    default:
      sosfiltfilt_kernel<TIn, 0><<<grid, threads, smem, st>>>(x, rows, T, xs, group_rows, group_stride, a, y, ys);
  }
  count_launch();
  return cudaGetLastError();
}

cudaError_t sosfiltfilt_launch_grouped(const void* x, int x_is_f32, long rows, long T, long xs, int group_rows,
                                       long group_stride, const SosArgs& a, double* y, long ys, cudaStream_t st) {
  if (x_is_f32) return sos_launch_t<float>((const float*)x, rows, T, xs, group_rows, group_stride, a, y, ys, st);
  return sos_launch_t<double>((const double*)x, rows, T, xs, group_rows, group_stride, a, y, ys, st);
}

cudaError_t sosfiltfilt_launch(const void* x, int x_is_f32, long rows, long T, long xs, const SosArgs& a, double* y,
                               long ys, cudaStream_t st) {
  // a single group: row r at x + r*xs
  return sosfiltfilt_launch_grouped(x, x_is_f32, rows, T, xs, (int)(rows > 0x7fffffffL ? 0x7fffffff : rows), 0, a, y,
                                    ys, st);
}

// ---------------------------------------------------------------------------
// K5: derivative along time of the filtered MFCC rows and the norm over rows
// (script/mfcc.py:405-415).  One thread per (clip, frame), coalesced along time.
// ---------------------------------------------------------------------------
__global__ void delta_norm_kernel(const double* __restrict__ x, int rows, long T, int method,
                                  double* __restrict__ tot) {
  const long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  const long clip = blockIdx.y;
  const double* base = x + (size_t)clip * rows * T;
  double s = 0.0;
  for (int r = 0; r < rows; ++r) {
    const double* f = base + (size_t)r * T;
    double d;
    if (T == 1) {
      d = 0.0;
    } else if (t == 0) {
      d = (method == 0 || T < 3) ? f[1] - f[0] : (-3.0 * f[0] + 4.0 * f[1] - f[2]) / 2.0;
    } else if (t == T - 1) {
      d = (method == 0 || T < 3) ? f[T - 1] - f[T - 2] : (3.0 * f[T - 1] - 4.0 * f[T - 2] + f[T - 3]) / 2.0;
    } else {
      d = (f[t + 1] - f[t - 1]) / 2.0;
    }
    s += d * d;
  }
  tot[(size_t)clip * T + t] = sqrt(s) / (double)rows;
}

cudaError_t delta_norm_launch(const double* x, long n_clips, int rows, long T, int method, double* tot,
                              cudaStream_t st) {
  dim3 grid((unsigned)((T + 255) / 256), (unsigned)n_clips);
  delta_norm_kernel<<<grid, 256, 0, st>>>(x, rows, T, method, tot);
  count_launch();
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// scipy.signal.filtfilt(b, 1, x): zero-phase FIR.  With a == 1 the lfilter
// initial state zi*x[0] is "the past was constantly x[0]", so each pass is a
// plain convolution over the odd-extended signal with a constant extension
// beyond its first sample -- no recurrence, one thread per output.
// ---------------------------------------------------------------------------
__device__ __forceinline__ double odd_ext_at(const double* xr, long T, int p, long i) {
  if (i < p) return 2.0 * xr[0] - xr[p - i];
  if (i < p + T) return xr[i - p];
  return 2.0 * xr[T - 1] - xr[T - 2 - (i - p - T)];
}

__global__ void fir_fwd_kernel(const double* __restrict__ x, long T, int p, const double* __restrict__ b, int n_taps,
                               double* __restrict__ work) {
  const long L = T + 2L * p;
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= L) return;
  const double* xr = x + (size_t)blockIdx.y * T;
  double acc = 0.0;
  for (int j = n_taps - 1; j >= 0; --j) {
    const long m = i - j;
    acc = fma(b[j], odd_ext_at(xr, T, p, m < 0 ? 0 : m), acc);
  }
  work[(size_t)blockIdx.y * L + i] = acc;
}

__global__ void fir_bwd_kernel(const double* __restrict__ work, long T, int p, const double* __restrict__ b,
                               int n_taps, double* __restrict__ y) {
  const long L = T + 2L * p;
  const long n = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= T) return;
  const double* w = work + (size_t)blockIdx.y * L;
  const long i = n + p;
  double acc = 0.0;
  for (int j = n_taps - 1; j >= 0; --j) {
    const long m = i + j;
    acc = fma(b[j], w[m >= L ? L - 1 : m], acc);
  }
  y[(size_t)blockIdx.y * T + n] = acc;
}

cudaError_t fir_filtfilt_launch(const double* x, long rows, long T, const double* b_dev, int n_taps, double* y,
                                double* work, cudaStream_t st) {
  const int p = 3 * n_taps;
  const long L = T + 2L * p;
  dim3 g1((unsigned)((L + 255) / 256), (unsigned)rows), g2((unsigned)((T + 255) / 256), (unsigned)rows);
  fir_fwd_kernel<<<g1, 256, 0, st>>>(x, T, p, b_dev, n_taps, work);
  fir_bwd_kernel<<<g2, 256, 0, st>>>(work, T, p, b_dev, n_taps, y);
  count_launch(2);
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// Banded stencil with dense boundary rows (np.gradient / savgol 'interp' /
// findiff; script/calc.py:635-645, script/mfcc.py:130).
// ---------------------------------------------------------------------------
__global__ void stencil_kernel(const double* __restrict__ x, long T, const double* __restrict__ coef, int half,
                               const double* __restrict__ el, const double* __restrict__ er, int n_edge,
                               int n_edge_in, double* __restrict__ y) {
  const long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  const double* xr = x + (size_t)blockIdx.y * T;
  double acc = 0.0;
  if (t < n_edge) {
    for (int i = 0; i < n_edge_in; ++i) acc = fma(el[t * n_edge_in + i], xr[i], acc);
  } else if (t >= T - n_edge) {
    const long q = t - (T - n_edge);
    for (int i = 0; i < n_edge_in; ++i) acc = fma(er[q * n_edge_in + i], xr[T - n_edge_in + i], acc);
  } else {
    for (int o = -half; o <= half; ++o) acc = fma(coef[o + half], xr[t + o], acc);
  }
  y[(size_t)blockIdx.y * T + t] = acc;
}

cudaError_t stencil_launch(const double* x, long rows, long T, const double* coef_dev, int half, const double* el_dev,
                           const double* er_dev, int n_edge, int n_edge_in, double* y, cudaStream_t st) {
  dim3 grid((unsigned)((T + 255) / 256), (unsigned)rows);
  stencil_kernel<<<grid, 256, 0, st>>>(x, T, coef_dev, half, el_dev, er_dev, n_edge, n_edge_in, y);
  count_launch();
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// K6: modulation spectrum of the MFCC trajectories (SURVEY.md Appendix B).
// One CTA per (window, clip); each warp transforms one coefficient's window at a
// time: mean removal (shuffle reduction), periodic Hann, zero padding, radix-2
// FFT in shared memory (float64 arithmetic: magnitudes reach 1e3 and the parity
// budget is 1e-3 absolute), |X| out, and per-band energies reduced with warp
// shuffles into per-warp shared accumulators, summed in warp order at the end so
// that the result does not depend on which warp finishes first.
// ---------------------------------------------------------------------------
constexpr int kModWarps = 4;  // at most; fewer when the warps' FFT buffers would not fit (nfft 4096)
constexpr int kMaxBands = 16;
constexpr size_t kModSmem = 220 * 1024;

__global__ void __launch_bounds__(kModWarps * 32)
    modspec_kernel(const float* __restrict__ mfcc, int n_coef, long T, int win, int hop, int nfft, int log2n,
                   long n_win, float* __restrict__ mag, float* __restrict__ band, const int* __restrict__ band_lo,
                   const int* __restrict__ band_hi, int n_bands) {
  extern __shared__ __align__(16) unsigned char sm_raw[];
  const int n_warps = blockDim.x >> 5;
  double2* s_tw = reinterpret_cast<double2*>(sm_raw);           // [nfft/2]
  double2* s_buf = s_tw + nfft / 2;                             // [n_warps][nfft]
  double* s_hann = reinterpret_cast<double*>(s_buf + n_warps * nfft);  // [win]
  __shared__ double s_band[kModWarps][kMaxBands];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long j = blockIdx.x;   // window
  const long clip = blockIdx.y;
  const int nb = nfft / 2 + 1;

  for (int i = tid; i < nfft / 2; i += blockDim.x) {
    double s, c;
    sincospi(-2.0 * (double)i / (double)nfft, &s, &c);
    s_tw[i] = make_double2(c, s);
  }
  for (int i = tid; i < win; i += blockDim.x) s_hann[i] = 0.5 - 0.5 * cospi(2.0 * (double)i / (double)win);
  for (int i = tid; i < kModWarps * kMaxBands; i += blockDim.x) s_band[i / kMaxBands][i % kMaxBands] = 0.0;
  __syncthreads();

  double2* buf = s_buf + warp * nfft;
  for (int c = warp; c < n_coef; c += n_warps) {
    const float* src = mfcc + ((size_t)clip * n_coef + c) * T + j * hop;
    double sum = 0.0;
    for (int i = lane; i < win; i += 32) sum += (double)src[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const double mean = sum / (double)win;
    for (int i = lane; i < nfft; i += 32) {
      const double v = i < win ? ((double)src[i] - mean) * s_hann[i] : 0.0;
      buf[__brev((unsigned)i) >> (32 - log2n)] = make_double2(v, 0.0);
    }
    __syncwarp();
    for (int s = 0; s < log2n; ++s) {
      const int half = 1 << s;
      const int tw_step = nfft >> (s + 1);
      for (int bfly = lane; bfly < nfft / 2; bfly += 32) {
        const int pos = bfly & (half - 1);
        const int i0 = ((bfly >> s) << (s + 1)) + pos, i1 = i0 + half;
        const double2 w = s_tw[pos * tw_step];
        const double2 u = buf[i0], v = buf[i1];
        const double2 tv = make_double2(v.x * w.x - v.y * w.y, v.x * w.y + v.y * w.x);
        buf[i0] = make_double2(u.x + tv.x, u.y + tv.y);
        buf[i1] = make_double2(u.x - tv.x, u.y - tv.y);
      }
      __syncwarp();
    }
    float* mdst = mag != nullptr ? mag + (((size_t)clip * n_coef + c) * n_win + j) * nb : nullptr;
    for (int k = lane; k < nb; k += 32) {
      const double2 X = buf[k];
      const double p = X.x * X.x + X.y * X.y;
      if (mdst) mdst[k] = (float)sqrt(p);
    }
    if (band != nullptr) {
      for (int b = 0; b < n_bands; ++b) {
        double e = 0.0;
        for (int k = band_lo[b] + lane; k < band_hi[b]; k += 32) {
          const double2 X = buf[k];
          e += X.x * X.x + X.y * X.y;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) e += __shfl_xor_sync(0xffffffffu, e, o);
        if (lane == 0) s_band[warp][b] += e;
      }
    }
    __syncwarp();
  }
  __syncthreads();
  if (band != nullptr && tid < n_bands) {
    double acc = 0.0;
    for (int w = 0; w < n_warps; ++w) acc += s_band[w][tid];
    band[((size_t)clip * n_win + j) * n_bands + tid] = (float)acc;
  }
}

cudaError_t modspec_launch(const float* mfcc, long n_clips, int n_coef, long T, int win, int hop, int nfft, float* mag,
                           float* band, const int* band_lo_dev, const int* band_hi_dev, int n_bands, cudaStream_t st) {
  int log2n = 0;
  while ((1 << log2n) < nfft) ++log2n;
  const long n_win = T >= win ? 1 + (T - win) / hop : 0;
  if (n_win <= 0) return cudaSuccess;
  // warps per CTA from the shared-memory budget: each holds one nfft-point complex fp64 buffer (nfft 4096: 2 warps,
  // 192 KB)
  const size_t fixed = (size_t)(nfft / 2) * 16 + (size_t)win * 8;
  const size_t per_warp = (size_t)nfft * 16;
  const int warps = fixed + kModWarps * per_warp <= kModSmem ? kModWarps : (int)((kModSmem - fixed) / per_warp);
  const size_t smem = fixed + (size_t)warps * per_warp;
  cudaError_t e = cudaFuncSetAttribute(modspec_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kModSmem);
  if (e != cudaSuccess) return e;
  // grid.y is limited to 65535: fold clips beyond that into several launches
  for (long c0 = 0; c0 < n_clips; c0 += 65535) {
    const long nc = n_clips - c0 < 65535 ? n_clips - c0 : 65535;
    dim3 grid((unsigned)n_win, (unsigned)nc);
    modspec_kernel<<<grid, warps * 32, smem, st>>>(
        mfcc + (size_t)c0 * n_coef * T, n_coef, T, win, hop, nfft, log2n, n_win,
        mag ? mag + (size_t)c0 * n_coef * n_win * (nfft / 2 + 1) : nullptr,
        band ? band + (size_t)c0 * n_win * n_bands : nullptr, band_lo_dev, band_hi_dev, n_bands);
    count_launch();
  }
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// Ragged RMS envelope (librosa.feature.rms, pad_mode='constant'; script/calc.py:326-331) of packed clips.  Each frame
// is one warp's sum: lane l accumulates fmaf(v, v, s) over i = l, l + 32, ... from 0, samples outside [0, len) read as
// 0, then the xor-shuffle tree 16, 8, 4, 2, 1 and sqrtf(s / frame_length).  That order is the contract: every output's
// bits are fixed by it, whatever chunk or batch the clip sits in (a running sum over the hop would be cheaper and
// would change them).  A work item (one CTA) is F consecutive frames of one clip (RmsClip); its span of
// (F - 1) * hop + frame_length samples is read from global memory once, int16 scaled on load as pcm16_to_f32_kernel
// scales it, into shared memory, where the overlapping frames (10x at 0.1 s / 0.01 s) find it.  A clip whose frame
// alone is over kRmsSpan reads its frames from global memory in the same order.
// ---------------------------------------------------------------------------
template <typename X>
__global__ void __launch_bounds__(kRmsWarps * 32) rms_varlen_kernel(const X* __restrict__ x,
                                                                     const RmsClip* __restrict__ clips,
                                                                     const unsigned* __restrict__ first_item,
                                                                     long n_clips, float* __restrict__ out) {
  __shared__ float xs[kRmsSpan];
  constexpr float kq = 1.0f / 32768.0f;
  const unsigned item = blockIdx.x;
  long clip = 0, hi_c = n_clips - 1;  // the clip owning this item: the last with first_item[clip] <= item
  while (clip < hi_c) {
    const long mid = (clip + hi_c + 1) >> 1;
    if (first_item[mid] <= item) clip = mid;
    else hi_c = mid - 1;
  }
  const RmsClip c = clips[clip];
  const X* xr = x + c.src;
  auto ld = [&](long m) -> float {
    if (m < 0 || m >= c.len) return 0.0f;
    if constexpr (sizeof(X) == 2) return (float)xr[m] * kq;
    else return xr[m];
  };
  const long f0 = (long)(item - first_item[clip]) * c.F;
  const int nf = (int)min((long)c.F, c.T - f0);
  const long start0 = f0 * c.hop - c.pad;
  const bool staged = (long)(c.F - 1) * c.hop + c.frame_length <= kRmsSpan;  // the same for every item of the clip
  if (staged) {
    const int span = (nf - 1) * c.hop + c.frame_length;
    for (int j = threadIdx.x; j < span; j += kRmsWarps * 32) xs[j] = ld(start0 + j);
    __syncthreads();
  }
  const int lane = threadIdx.x & 31;
  for (int f = threadIdx.x >> 5; f < nf; f += kRmsWarps) {
    float s = 0.0f;
    if (staged) {
      const float* w = xs + f * c.hop;
      for (int i = lane; i < c.frame_length; i += 32) {
        const float v = w[i];
        s = fmaf(v, v, s);
      }
    } else {
      const long start = start0 + (long)f * c.hop;
      for (int i = lane; i < c.frame_length; i += 32) {
        const float v = ld(start + i);
        s = fmaf(v, v, s);
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) out[c.out + f0 + f] = sqrtf(s / (float)c.frame_length);
  }
}

cudaError_t rms_varlen_launch(const void* x, int pcm16, const RmsClip* clips, const unsigned* first_item, long n_clips,
                              long n_items, float* out, cudaStream_t st) {
  if (pcm16)
    rms_varlen_kernel<<<(unsigned)n_items, kRmsWarps * 32, 0, st>>>((const int16_t*)x, clips, first_item, n_clips, out);
  else
    rms_varlen_kernel<<<(unsigned)n_items, kRmsWarps * 32, 0, st>>>((const float*)x, clips, first_item, n_clips, out);
  count_launch();
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// PCM16 ingest: what librosa.load does to a 16-bit WAV before the path starts
// (script/mfcc.py:373 -> soundfile -> float32 = int16 / 32768), on the device, so that
// only 2 bytes per sample cross PCIe.  8 samples per thread, 128-bit accesses.
// ---------------------------------------------------------------------------
__global__ void pcm16_to_f32_kernel(const int16_t* __restrict__ x, long n, float* __restrict__ y) {
  const long i8 = ((long)blockIdx.x * blockDim.x + threadIdx.x) * 8;
  constexpr float k = 1.0f / 32768.0f;
  if (i8 + 8 <= n && (reinterpret_cast<uintptr_t>(x + i8) & 15) == 0 && (reinterpret_cast<uintptr_t>(y + i8) & 15) == 0) {
    const int4 v = *reinterpret_cast<const int4*>(x + i8);
    const int w[4] = {v.x, v.y, v.z, v.w};
    float o[8];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      o[2 * q] = (float)(short)(w[q] & 0xffff) * k;
      o[2 * q + 1] = (float)(short)(w[q] >> 16) * k;
    }
    *reinterpret_cast<float4*>(y + i8) = make_float4(o[0], o[1], o[2], o[3]);
    *reinterpret_cast<float4*>(y + i8 + 4) = make_float4(o[4], o[5], o[6], o[7]);
  } else {
    for (long i = i8; i < n && i < i8 + 8; ++i) y[i] = (float)x[i] * k;
  }
}

cudaError_t pcm16_to_f32_launch(const int16_t* x, long n, float* y, cudaStream_t st) {
  const long threads = (n + 7) / 8;
  pcm16_to_f32_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(x, n, y);
  count_launch();
  return cudaGetLastError();
}

// Padded rows -> packed blocks.  Clip i owns `rows` rows of cnt[i] * unit elements, the first at
// src + i * rows * pitch, the next `pitch` elements on; they leave back to back at dst + off[i] * rows * unit.  One CTA
// per (clip, row); a plain copy, so the bits are kept.
template <typename E>
__global__ void compact_rows_kernel(const E* __restrict__ src, E* __restrict__ dst, int rows, int unit, long pitch,
                                    const int* __restrict__ cnt, const long* __restrict__ off) {
  const long clip = blockIdx.x / rows;
  const int r = (int)(blockIdx.x - clip * rows);
  const long len = (long)cnt[clip] * unit;
  const E* s = src + ((size_t)clip * rows + r) * pitch;
  E* d = dst + ((size_t)off[clip] * rows + (size_t)r * cnt[clip]) * unit;
  for (long e = threadIdx.x; e < len; e += blockDim.x) d[e] = s[e];
}

cudaError_t compact_rows_launch(const void* src, void* dst, int elem_bytes, long n_clips, int rows, int unit,
                                long pitch, const int* cnt, const long* off, cudaStream_t st) {
  const unsigned grid = (unsigned)(n_clips * rows);
  if (elem_bytes == 8)
    compact_rows_kernel<<<grid, 256, 0, st>>>((const double*)src, (double*)dst, rows, unit, pitch, cnt, off);
  else
    compact_rows_kernel<<<grid, 256, 0, st>>>((const float*)src, (float*)dst, rows, unit, pitch, cnt, off);
  count_launch();
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// Ragged, multi-ratio polyphase resampler with scipy.signal.resample_poly / upfirdn semantics
// (the step before the path: librosa.load(sr=sigSr) at script/mfcc.py:373, :284).  For each clip,
//   y_full[m] = sum_i h[m*down - i*up] * x[i],  y = y_full[n_pre_remove : n_pre_remove + n_out],
// each output one float64 fma chain over i ascending from i_lo to i_hi (the bounds below, from the clip's own len_h).
// That order is the contract: every output's bits are fixed by it, whatever the layout of taps and samples.
// A work item is kRsOut consecutive outputs of one clip, one per thread.  Its input span goes through shared memory in
// coalesced tiles (int16 scaled on load, as pcm16_to_f32_kernel scales it); one tile holds the span of every ratio
// whose 256 outputs need at most kRsTile inputs (all the usual audio rates), more tiles walk i in order.  The tap
// table in its natural order is already polyphase (tap j of phase p at j * up + p): at each step of the chain, the
// threads of a warp away from the clip's edges read taps within one window of about 2 * up floats, from L1.  Plan-rate
// clips (copy) are staged as the packed host path always staged them: x, or (float)x / 32768 for int16, in the same
// launch.
// ---------------------------------------------------------------------------
constexpr int kRsTile = 4096;

template <typename X>
__global__ void __launch_bounds__(kRsOut) resample_rows_kernel(const X* __restrict__ x, const RsClip* __restrict__ clips,
                                                               const unsigned* __restrict__ first_item, long n_clips,
                                                               const float* __restrict__ hp, float* __restrict__ y,
                                                               long y_stride) {
  __shared__ float xs[kRsTile];
  constexpr float kq = 1.0f / 32768.0f;
  const unsigned item = blockIdx.x;
  long clip = 0, hi_c = n_clips - 1;  // the clip owning this item: the last with first_item[clip] <= item
  while (clip < hi_c) {
    const long mid = (clip + hi_c + 1) >> 1;
    if (first_item[mid] <= item) clip = mid;
    else hi_c = mid - 1;
  }
  const RsClip c = clips[clip];
  const X* xr = x + c.src;
  float* yr = y + clip * y_stride;
  const long m0 = (long)(item - first_item[clip]) * kRsOut, mo = m0 + threadIdx.x;
  const long m_last = min(m0 + kRsOut, c.n_out) - 1;
  auto ld = [&](long i) -> float {
    if constexpr (sizeof(X) == 2) return (float)xr[i] * kq;
    else return xr[i];
  };
  if (c.copy) {
    if (mo <= m_last) yr[mo] = ld(mo);
    return;
  }
  // i_hi: largest i with pos - i*up >= 0; i_lo: smallest i with pos - i*up <= len_h - 1
  auto lo_of = [&](long pos) { return pos - c.len_h + 1 <= 0 ? 0L : (pos - c.len_h + c.up) / c.up; };
  auto hi_of = [&](long pos) { return min(pos / c.up, c.n_in - 1); };
  const long pos = (min(mo, m_last) + c.n_pre_remove) * c.down;  // position in the zero-stuffed input
  const long q = pos / c.up;
  long i_lo = lo_of(pos), i_hi = hi_of(pos);
  if (mo > m_last) i_lo = 1, i_hi = 0;
  const long I0 = lo_of((m0 + c.n_pre_remove) * c.down), I1 = hi_of((m_last + c.n_pre_remove) * c.down);
  const float* h = hp + c.tap0 + (pos - q * c.up);  // this output's phase: h[k] at h[(q - i) * up]
  double acc = 0.0;
  for (long t0 = I0; t0 <= I1; t0 += kRsTile) {
    const long t1 = min(t0 + kRsTile, I1 + 1);
    __syncthreads();
    for (long i = t0 + threadIdx.x; i < t1; i += kRsOut) xs[i - t0] = ld(i);
    __syncthreads();
    const long a = max(i_lo, t0), b = min(i_hi, t1 - 1);
    if (a > b) continue;
    const float* hj = h + (q - a) * c.up;
    const float* xi = xs + (a - t0);
    const int n = (int)(b - a + 1);
#pragma unroll 4
    for (int s = 0; s < n; ++s) acc = fma((double)hj[-(long)s * c.up], (double)xi[s], acc);
  }
  if (mo <= m_last) yr[mo] = (float)acc;
}

cudaError_t resample_rows_launch(const void* x, int pcm16, const RsClip* clips, const unsigned* first_item,
                                 long n_clips, long n_items, const float* h_poly, float* y, long y_stride,
                                 cudaStream_t st) {
  if (pcm16)
    resample_rows_kernel<<<(unsigned)n_items, kRsOut, 0, st>>>((const int16_t*)x, clips, first_item, n_clips, h_poly,
                                                               y, y_stride);
  else
    resample_rows_kernel<<<(unsigned)n_items, kRsOut, 0, st>>>((const float*)x, clips, first_item, n_clips, h_poly, y,
                                                               y_stride);
  count_launch();
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// Local maxima of each row with scipy.signal.find_peaks' default semantics (the step after the
// path: script/main.py:1566, :1601 and script/calc.py:669, :681 call find_peaks(+-curve)):
// a peak is a sample, or a flat run of equal samples, strictly higher than both neighbours;
// a flat run reports its middle index (left + right) / 2; the first and last sample never are.
// One warp per row; peaks come out in ascending order (ballot + prefix popcount).  `sign` = -1
// finds minima.  count[row] holds the total number found even when it exceeds max_peaks.
// ---------------------------------------------------------------------------
__global__ void find_peaks_kernel(const double* __restrict__ x, long rows, long T, long stride, double sign,
                                  int max_peaks, int* __restrict__ idx, int* __restrict__ count) {
  const long row = ((long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const double* xr = x + row * stride;
  int* out = idx + row * (long)max_peaks;
  int base = 0;
  for (long t0 = 1; t0 < T - 1; t0 += 32) {
    const long t = t0 + lane;
    bool is_peak = false;
    int where = 0;
    if (t < T - 1) {
      const double v = sign * xr[t];
      if (sign * xr[t - 1] < v) {  // rising edge: the run starting here may be a peak
        long r = t;
        while (r + 1 < T && sign * xr[r + 1] == v) ++r;
        if (r + 1 < T && sign * xr[r + 1] < v) {
          is_peak = true;
          where = (int)((t + r) / 2);
        }
      }
    }
    const unsigned mask = __ballot_sync(0xffffffffu, is_peak);
    if (is_peak) {
      const int pos = base + __popc(mask & ((1u << lane) - 1u));
      if (pos < max_peaks) out[pos] = where;
    }
    base += __popc(mask);
  }
  if (lane == 0) count[row] = base;
}

cudaError_t find_peaks_launch(const double* x, long rows, long T, long stride, int minima, int max_peaks, int* idx,
                              int* count, cudaStream_t st) {
  const long threads = rows * 32;
  find_peaks_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(x, rows, T, stride, minima ? -1.0 : 1.0, max_peaks,
                                                                     idx, count);
  count_launch();
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// Hilbert envelope |scipy.signal.hilbert(x)| (script/calc.py:284-286, script/mfcc.py 'Hilb').
// scipy zeroes the negative frequencies of an N-point FFT; for real x that is x + i*y with y the
// CIRCULAR convolution of x with the discrete Hilbert kernel
//   g[k] = (1/N) * (cos(pi k/N) - (-1)^k [* cos(pi k/N) if N even]) / sin(pi k/N),  g[0] = 0
// (N even: 2/N * cot(pi k/N) for odd k, 0 for even k).  N is arbitrary (e.g. 160 000), so instead
// of an arbitrary-length FFT the convolution is evaluated directly: N^2 FMAs (2.6e10 for a 10 s
// clip, about a millisecond of B200 FP32) with the classic register-blocked shared-memory FIR
// tiling -- same result as scipy's FFT formulation to float32 rounding.
// ---------------------------------------------------------------------------
__global__ void hilbert_kernel_table(long n, float* __restrict__ g) {
  const long k = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  if (k == 0) {
    g[0] = 0.0f;
    return;
  }
  double s, c;
  sincospi((double)k / (double)n, &s, &c);
  const double sign = (k & 1) ? -1.0 : 1.0;
  const double num = (n & 1) ? (c - sign) : (c - sign * c);
  g[k] = (float)(num / ((double)n * s));
}

constexpr int kHilThreads = 256;
constexpr int kHilR = 8;                        // consecutive outputs per thread
constexpr int kHilTN = kHilThreads * kHilR;     // outputs per block
constexpr int kHilTK = 512;                     // taps per shared-memory chunk

// partial[ks][n] = sum over k in the ks-th slice of g[k] * x[(n - k) mod N]
__global__ void __launch_bounds__(kHilThreads)
    hilbert_conv_kernel(const float* __restrict__ x, const float* __restrict__ g, long n, int ksplit,
                        double* __restrict__ partial) {
  __shared__ __align__(16) float sg[kHilTK];
  __shared__ __align__(16) float sx[kHilTN + kHilTK];
  const int tid = threadIdx.x;
  const long n0 = (long)blockIdx.x * kHilTN;
  const int ks = blockIdx.y;
  const long k_per = ((n + ksplit - 1) / ksplit + kHilTK - 1) / kHilTK * kHilTK;
  const long k_lo = (long)ks * k_per, k_hi = min(n, k_lo + k_per);
  double acc[kHilR];
#pragma unroll
  for (int r = 0; r < kHilR; ++r) acc[r] = 0.0;
  for (long k0 = k_lo; k0 < k_hi; k0 += kHilTK) {
    __syncthreads();
    for (int i = tid; i < kHilTK; i += kHilThreads) sg[i] = (k0 + i < k_hi) ? g[k0 + i] : 0.0f;
    // sx[i] = x[(n0 - k0 - (TK - 1) + i) mod N], i in [0, TN + TK - 1)
    for (int i = tid; i < kHilTN + kHilTK; i += kHilThreads) {
      long j = (n0 - k0 - (kHilTK - 1) + i) % n;
      if (j < 0) j += n;
      sx[i] = x[j];
    }
    __syncthreads();
    float a32[kHilR];
#pragma unroll
    for (int r = 0; r < kHilR; ++r) a32[r] = 0.0f;
    // output n0 + tid*8 + r, tap kk: x index in sx = tid*8 + r - kk + TK - 1
    const float* xb = sx + tid * kHilR + kHilTK - 8;
#pragma unroll 2
    for (int kk0 = 0; kk0 < kHilTK; kk0 += 8) {
      float w[16];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float4 v = *reinterpret_cast<const float4*>(xb - kk0 + 4 * q);
        w[4 * q] = v.x;
        w[4 * q + 1] = v.y;
        w[4 * q + 2] = v.z;
        w[4 * q + 3] = v.w;
      }
      const float4 g0 = *reinterpret_cast<const float4*>(sg + kk0), g1 = *reinterpret_cast<const float4*>(sg + kk0 + 4);
      const float gg[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
#pragma unroll
      for (int u = 0; u < 8; ++u)
#pragma unroll
        for (int r = 0; r < kHilR; ++r) a32[r] = fmaf(gg[u], w[r - u + 7], a32[r]);
    }
#pragma unroll
    for (int r = 0; r < kHilR; ++r) acc[r] += (double)a32[r];
  }
#pragma unroll
  for (int r = 0; r < kHilR; ++r) {
    const long nn = n0 + (long)tid * kHilR + r;
    if (nn < n) partial[(size_t)ks * n + nn] = acc[r];
  }
}

__global__ void hilbert_finish_kernel(const float* __restrict__ x, const double* __restrict__ partial, long n, int ksplit,
                                      float* __restrict__ amp) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double y = 0.0;
  for (int ks = 0; ks < ksplit; ++ks) y += partial[(size_t)ks * n + i];
  const double xv = (double)x[i];
  amp[i] = (float)sqrt(xv * xv + y * y);
}

cudaError_t hilbert_envelope_launch(const float* x, long n_clips, long n, long stride, float* amp, long amp_stride,
                                    int sm_count, cudaStream_t st) {
  float* g = nullptr;
  double* partial = nullptr;
  const int n_blocks = (int)((n + kHilTN - 1) / kHilTN);
  int ksplit = (2 * sm_count + n_blocks - 1) / n_blocks;
  const int max_split = (int)((n + kHilTK - 1) / kHilTK);
  ksplit = ksplit < 1 ? 1 : (ksplit > max_split ? max_split : (ksplit > 64 ? 64 : ksplit));
  cudaError_t e;
  if ((e = cudaMallocAsync((void**)&g, (size_t)n * 4, st)) != cudaSuccess) return e;
  if ((e = cudaMallocAsync((void**)&partial, (size_t)ksplit * n * 8, st)) != cudaSuccess) {
    cudaFreeAsync(g, st);
    return e;
  }
  hilbert_kernel_table<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(n, g);
  count_launch();
  for (long c = 0; c < n_clips; ++c) {
    hilbert_conv_kernel<<<dim3((unsigned)n_blocks, (unsigned)ksplit), kHilThreads, 0, st>>>(x + c * stride, g, n, ksplit,
                                                                                          partial);
    hilbert_finish_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(x + c * stride, partial, n, ksplit,
                                                                       amp + c * amp_stride);
    count_launch(2);
  }
  e = cudaGetLastError();
  cudaFreeAsync(g, st);
  cudaFreeAsync(partial, st);
  return e;
}

__global__ void fill_i32_kernel(int* p, long n, int v) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}
cudaError_t fill_i32_launch(int* p, long n, int v, cudaStream_t st) {
  fill_i32_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(p, n, v);
  count_launch();
  return cudaGetLastError();
}

}  // namespace mmf
